// orb.cu — B200 (sm_100a) ORB extractor: pyramid / FAST+NMS / octree distribution / IC orientation /
// 7x7 blur / rBRIEF-256, batched over frames.  Replaces ORBextractor (reference src/ORBextractor.cc).
//
// Everything stays in HBM between the frame upload and the keypoint/descriptor download:
//   k_resize      (x L-1)  level l-1 -> l, cv::resize(INTER_LINEAR) fixed-point          ORBextractor.cc:1107-1132
//   k_fast                 one CTA per 30-px cell: FAST-9-16 score, in-cell NMS, 20/7 rule ORBextractor.cc:789-829
//   k_octree               one CTA per (level, frame): DistributeOctTree, array form       ORBextractor.cc:539-763
//   k_blur                 7x7 sigma-2 fixed-point Gaussian of every level                 ORBextractor.cc:1085-1086
//   k_orient_desc          one warp per keypoint: IC_Angle + rBRIEF + KeyPoint assembly    ORBextractor.cc:77-147,1043-1105
// Bit-exactness notes: all float work uses explicit _rn intrinsics (no FMA contraction); cos/sin are
// evaluated in double and narrowed (canonical correctly-rounded f32, SURVEY.md 7.3 item 4).
#include "common.cuh"
#include "mathx.cuh"
#include <cuda.h>
#include <cudaTypedefs.h>
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdlib>
#include <vector>

namespace sslpl {

constexpr int MAXL = SSLPL_MAX_LEVELS;
constexpr int EDGE = 19;            // EDGE_THRESHOLD, ORBextractor.cc:74
constexpr int MINB = EDGE - 3;      // minBorderX/Y, ORBextractor.cc:775
constexpr int HALF_PATCH = 15;
constexpr int BLUR_TW = 64, BLUR_TH = 32;

struct LevelGeom {
    int w, h, pitch;                 // level image (level 0: the input view's pitch is used instead)
    long long img_off;               // byte offset inside the per-frame pyramid block (levels >= 1)
    int bpitch; long long blur_off;  // blurred plane inside the per-frame blur block
    int nCols, nRows, wCell, hCell, maxBX, maxBY;
    int cell_base, ncells, cell_cap;
    long long cand_off;              // u32 offset inside the per-frame candidate block
    int key_cap; long long key_off;  // offset inside the per-frame key arrays
    int nfeat, kp_cap, kp_base;
    int pool_cap; long long pool_off;
    int xtab_off, ytab_off;          // resize tables (int2 entries)
    int tile_base, tiles_x, tiles_y; // blur tiles (64x32 over the whole level)
    float scale, patch_size;
};

struct OrbGeom {
    int nlevels, total_cells, total_tiles, kp_total_cap, iniTh, minTh, sort_cap;
    long long pyr_stride, blur_stride, cand_stride, key_stride, pool_stride;
    int umax[16];
    LevelGeom lv[MAXL];
};

struct OrbWs {
    uint8_t* pyr; uint8_t* blur;
    uint32_t* cand; int* cell_cnt; int* cell_off;
    uint32_t* kxyr; int* knode;
    short4* nbox; int* ncnt; int* nq; uint8_t* nalive; unsigned* nbest; int* scan; int* ord;
    uint32_t* lvl_kp; int* lvl_cnt;
    int2* rtab;
    int* err;
    sslpl_keypoint* kps; uint8_t* desc; int* nkp;
    CUtensorMap* tmaps;          // MAXL tensor maps in global memory (64-byte aligned)
};

struct View { const uint8_t* base; int pitch; long long frame_stride; };

__constant__ signed char c_pattern[1024] = {
#include "orb_pattern.inc"
};

__device__ __forceinline__ const uint8_t* level_ptr(const OrbGeom& g, const OrbWs& ws, const View& v, int level, int frame, int* pitch) {
    if (level == 0) { *pitch = v.pitch; return v.base + (long long)frame * v.frame_stride; }
    *pitch = g.lv[level].pitch;
    return ws.pyr + (long long)frame * g.pyr_stride + g.lv[level].img_off;
}

// ------------------------------------------------------------------------------------------------
// cv::resize(INTER_LINEAR) 8UC1, 11-bit fixed point (SURVEY.md A.1); tables hold (sx, a0 | a1<<16)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_resize(const __grid_constant__ OrbGeom g, OrbWs ws, View v, int level) {
    const LevelGeom& d = g.lv[level];
    const LevelGeom& s = g.lv[level - 1];
    const int x4 = (blockIdx.x * 32 + threadIdx.x) * 4, y = blockIdx.y * 8 + threadIdx.y, f = blockIdx.z;
    if (y >= d.h || x4 >= d.w) return;
    int sp, dp;
    const uint8_t* S = level_ptr(g, ws, v, level - 1, f, &sp);
    uint8_t* D = const_cast<uint8_t*>(level_ptr(g, ws, v, level, f, &dp));
    const int2 ty = __ldg(&ws.rtab[d.ytab_off + y]);
    const int b0 = ty.y & 0xffff, b1 = ty.y >> 16;
    const uint8_t* S0 = S + (long long)ty.x * sp;
    const uint8_t* S1 = S + (long long)min(ty.x + 1, s.h - 1) * sp;
    uint32_t out = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int x = x4 + i;
        if (x < d.w) {
            const int2 tx = __ldg(&ws.rtab[d.xtab_off + x]);
            const int a0 = tx.y & 0xffff, a1 = tx.y >> 16, sx = tx.x, sx1 = min(sx + 1, s.w - 1);
            const int r0 = __ldg(S0 + sx) * a0 + __ldg(S0 + sx1) * a1;
            const int r1 = __ldg(S1 + sx) * a0 + __ldg(S1 + sx1) * a1;
            const int o = (((b0 * (r0 >> 4)) >> 16) + ((b1 * (r1 >> 4)) >> 16) + 2) >> 2;
            out |= (uint32_t)(o & 255) << (8 * i);
        }
    }
    uint8_t* dst = D + (long long)y * dp + x4;
    if (x4 + 3 < d.w) *reinterpret_cast<uint32_t*>(dst) = out;      // pitch and x4 are multiples of 4
    else for (int i = 0; x4 + i < d.w; i++) dst[i] = (uint8_t)(out >> (8 * i));
}

// ------------------------------------------------------------------------------------------------
// FAST-9-16 corner score (OpenCV cornerScore<16>), with floor t: returns score if >= t else 0.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int fast_score_tile(const uint8_t* p, int pitch, int t) {
    const int v = p[0];
    int d[25];
    d[0] = v - p[3 * pitch];      d[8] = v - p[-3 * pitch];
    d[4] = v - p[3];              d[12] = v - p[-3];
    {   // a 9-arc contains one pixel of every opposite pair
        bool br = (d[0] > t || d[8] > t) && (d[4] > t || d[12] > t);
        bool dk = (d[0] < -t || d[8] < -t) && (d[4] < -t || d[12] < -t);
        if (!br && !dk) return 0;
    }
    d[1] = v - p[3 * pitch + 1];   d[2] = v - p[2 * pitch + 2];   d[3] = v - p[pitch + 3];
    d[5] = v - p[-pitch + 3];      d[6] = v - p[-2 * pitch + 2];  d[7] = v - p[-3 * pitch + 1];
    d[9] = v - p[-3 * pitch - 1];  d[10] = v - p[-2 * pitch - 2]; d[11] = v - p[-pitch - 3];
    d[13] = v - p[pitch - 3];      d[14] = v - p[2 * pitch - 2];  d[15] = v - p[3 * pitch - 1];
#pragma unroll
    for (int k = 16; k < 25; k++) d[k] = d[k - 16];
    int a0 = t;
#pragma unroll
    for (int k = 0; k < 16; k += 2) {
        int a = min(d[k + 1], d[k + 2]);
        a = min(a, d[k + 3]);
        if (a <= a0) continue;
        a = min(a, d[k + 4]); a = min(a, d[k + 5]); a = min(a, d[k + 6]); a = min(a, d[k + 7]); a = min(a, d[k + 8]);
        a0 = max(a0, min(a, d[k]));
        a0 = max(a0, min(a, d[k + 9]));
    }
    int b0 = -a0;
#pragma unroll
    for (int k = 0; k < 16; k += 2) {
        int b = max(d[k + 1], d[k + 2]);
        b = max(b, d[k + 3]);
        if (b >= b0) continue;
        b = max(b, d[k + 4]); b = max(b, d[k + 5]); b = max(b, d[k + 6]); b = max(b, d[k + 7]); b = max(b, d[k + 8]);
        b0 = min(b0, max(b, d[k]));
        b0 = min(b0, max(b, d[k + 9]));
    }
    const int s = -b0 - 1;
    return s >= t ? s : 0;
}

// ------------------------------------------------------------------------------------------------
// TMA / mbarrier helpers (sm_100a): one elected thread arms the barrier with the byte count and issues a
// cp.async.bulk.tensor.3d tile load (x, y, frame); out-of-bounds elements are zero-filled by the hardware.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok = 0;
    for (int spin = 0; !ok; spin++) {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}\n"
                     : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
        if (spin > (1 << 24)) __trap();          // never hang the box on a mis-programmed copy
    }
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* tm, int x, int y, int z, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(x), "r"(y), "r"(z), "r"(smem_u32(bar)) : "memory");
}

constexpr int TL_W = 64, TL_H = 32;            // output tile of the stencil kernels
constexpr int TL_P = 96, TL_IH = TL_H + 6;     // staged box: 96 x 38 bytes, origin (x0 - 16, y0 - 3).  For 1-byte elements TMA
                                               // requires the box to START on a 16-byte boundary in x (measured: tools/tma_probe.cu)
constexpr int TL_X = 16;                       // smem column of the tile's first output pixel

// Stage the 96x38 box of level `l`, frame `f` at (bx, by) into s_img (pitch TL_P).  TMA path: one bulk tensor copy,
// zero fill outside the level.  Fallback: aligned 32-bit loads (clamped to the row) or byte loads.
template <bool TMA>
__device__ __forceinline__ void stage_box(uint8_t* s_img, uint64_t* s_bar, const CUtensorMap* tm, const uint8_t* img, int pitch, int w, int h,
                                          int l, int f, int bx, int by) {
    const int tid = threadIdx.x;
    if (TMA) {
        if (tid == 0) { mbar_init(s_bar, 1); }
        __syncthreads();
        if (tid == 0) {
            // the descriptor lives in global memory and level 0 is rewritten by the host between launches
            asm volatile("fence.proxy.tensormap::generic.acquire.gpu [%0], 128;" ::"l"(reinterpret_cast<uint64_t>(tm + l)) : "memory");
            mbar_expect_tx(s_bar, TL_P * TL_IH);
            tma_load_3d(s_img, tm + l, bx, by, f, s_bar);
        }
        mbar_wait(s_bar, 0);
    } else {
        const bool al = ((reinterpret_cast<uintptr_t>(img) | (unsigned)pitch) & 3) == 0 && (bx & 3) == 0 && bx >= 0;
        if (al) {
            const int wmax = (pitch - bx) / 4 - 1;                       // last whole word of the row
            for (int i = tid; i < TL_IH * (TL_P / 4); i += blockDim.x) {
                const int r = i / (TL_P / 4), wi = i - r * (TL_P / 4);
                const int gy = min(max(by + r, 0), h - 1);
                const uint32_t v = __ldg(reinterpret_cast<const uint32_t*>(img + (long long)gy * pitch + bx) + min(wi, wmax));
                reinterpret_cast<uint32_t*>(s_img)[r * (TL_P / 4) + wi] = v;
            }
        } else {
            for (int i = tid; i < TL_IH * TL_P; i += blockDim.x) {
                const int r = i / TL_P, c = i - r * TL_P;
                const int gy = min(max(by + r, 0), h - 1), gx = min(max(bx + c, 0), w - 1);
                s_img[i] = __ldg(img + (long long)gy * pitch + gx);
            }
        }
        __syncthreads();
    }
}

constexpr int FAST_MAXC = 60;                 // wCell, hCell < 60 (ceil(w / floor(w/30)) < 60)
constexpr int FAST_TP = FAST_MAXC + 4;        // pitch of the per-cell score tile (1-px zero halo)
constexpr int FC_ROWS = 36 + TL_IH;           // staged rows: two 96x38 boxes, the second one 36 rows down (36*96 is a multiple of 128)

// One CTA per 30-px cell, the whole FAST stage in shared memory: stage the cell's (aw+6)x(ah+6) image box (TMA, the box
// starts on the 16-byte boundary at or before iniX), score it in two phases, in-cell NMS, 20/7 rule, ordered compaction.
//   phase A   the opposite-pair test on 4 pixels per thread with byte-SIMD video instructions; survivors are queued (~25 % of the pixels)
//   phase B1  the exact 9-arc corner test on 16-bit ring masks for the queued pixels; corners re-queued (~4 %)
//   phase B2  the full 16-ring score only for corners, all lanes busy; NMS walks the corner queue, survivors land in per-row bit masks
// Equivalent to the reference's per-cell cv::FAST(th=20) with fallback cv::FAST(th=7) (ORBextractor.cc:789-829): NMS
// inside the cell's detection area with outside pixels = 0, keep survivors >= iniTh or, if none, all survivors
// (SURVEY.md A.3 [probe]).  The detection areas of the cells are disjoint, so no pixel is scored twice and no score
// ever leaves the SM.
template <bool TMA>
__global__ void __launch_bounds__(128) k_fast(const __grid_constant__ OrbGeom g, OrbWs ws, View v, const CUtensorMap* tm) {
    __shared__ __align__(128) uint8_t s_img[FC_ROWS * TL_P];
    __shared__ __align__(4) uint8_t s_sc[(FAST_MAXC + 2) * FAST_TP];
    __shared__ unsigned short s_q[FAST_MAXC * FAST_MAXC];
    __shared__ unsigned long long s_rowall[FAST_MAXC], s_rowhi[FAST_MAXC];
    __shared__ int s_warp[33];
    __shared__ int s_qn, s_qc;
    __shared__ __align__(8) uint64_t s_bar;
    const int cell = blockIdx.x, f = blockIdx.y, tid = threadIdx.x, lane = tid & 31;
    int l = 0;
    while (l + 1 < g.nlevels && cell >= g.lv[l + 1].cell_base) l++;
    const LevelGeom& L = g.lv[l];
    const int ci = cell - L.cell_base, ci_i = ci / L.nCols, ci_j = ci - ci_i * L.nCols;
    int* cnt_out = ws.cell_cnt + (long long)f * g.total_cells + cell;
    const int iniX = MINB + ci_j * L.wCell, iniY = MINB + ci_i * L.hCell;
    const int maxX = min(iniX + L.wCell + 6, L.maxBX), maxY = min(iniY + L.hCell + 6, L.maxBY);
    const int cw = maxX - iniX, ch = maxY - iniY;
    if (iniX >= L.maxBX - 6 || iniY >= L.maxBY - 3 || cw < 7 || ch < 7) { if (tid == 0) *cnt_out = 0; return; }
    const int aw = cw - 6, ah = ch - 6, area = aw * ah;
    const int bx = iniX & ~15, xo = iniX + 3 - bx;          // smem column of the first detection pixel, 3..18
    int pitch;
    const uint8_t* img = level_ptr(g, ws, v, l, f, &pitch);
    const bool two = ch > TL_IH;
    if (TMA) {
        if (tid == 0) mbar_init(&s_bar, 1);
        __syncthreads();
        if (tid == 0) {
            asm volatile("fence.proxy.tensormap::generic.acquire.gpu [%0], 128;" ::"l"(reinterpret_cast<uint64_t>(tm + l)) : "memory");
            mbar_expect_tx(&s_bar, (two ? 2 : 1) * TL_P * TL_IH);
            tma_load_3d(s_img, tm + l, bx, iniY, f, &s_bar);
            if (two) tma_load_3d(s_img + 36 * TL_P, tm + l, bx, iniY + 36, f, &s_bar);   // rows 36, 37 arrive twice with the same bytes
        }
    } else {
        const bool al = ((reinterpret_cast<uintptr_t>(img) | (unsigned)pitch) & 3) == 0;
        const int rows = min(ch, FC_ROWS), wmax = (pitch - bx) / 4 - 1;
        if (al) {
            for (int i = tid; i < rows * (TL_P / 4); i += 128) {
                const int r = i / (TL_P / 4), wi = i - r * (TL_P / 4);
                reinterpret_cast<uint32_t*>(s_img)[i] =
                    __ldg(reinterpret_cast<const uint32_t*>(img + (long long)min(iniY + r, L.h - 1) * pitch + bx) + min(wi, wmax));
            }
        } else {
            for (int i = tid; i < rows * TL_P; i += 128) {
                const int r = i / TL_P, c = i - r * TL_P;
                s_img[i] = __ldg(img + (long long)min(iniY + r, L.h - 1) * pitch + min(bx + c, L.w - 1));
            }
        }
    }
    if (tid == 0) { s_qn = 0; s_qc = 0; }
    for (int i = tid; i < (ah + 2) * (FAST_TP / 4); i += 128) reinterpret_cast<uint32_t*>(s_sc)[i] = 0u;
    if (tid < FAST_MAXC) { s_rowall[tid] = 0ull; s_rowhi[tid] = 0ull; }
    if (TMA) mbar_wait(&s_bar, 0);
    __syncthreads();
    const int th = g.minTh;
    const unsigned ltmask = (1u << lane) - 1u;
    // phase A on the aligned word grid of the staged box: groups g0, g0+4, ... cover [xo, xo+aw)
    const unsigned T4 = 0x01010101u * (unsigned)th;
    const int g0 = xo & ~3, ng = (xo + aw - g0 + 3) >> 2, ngroups = ah * ng;
    const float inv_ng = __frcp_rn((float)ng);
    for (int gb = 0; gb < ngroups; gb += 128) {
        const int gidx = gb + tid;
        unsigned pm = 0;
        int r = 0, c4 = 0;
        if (gidx < ngroups) {
            r = __float2int_rz(__fmul_rn((float)gidx + 0.5f, inv_ng));                  // gidx / ng (exact: the quotient is >= 0.5/ng away from an integer)
            c4 = g0 + 4 * (gidx - r * ng);
            const unsigned* row = reinterpret_cast<const unsigned*>(&s_img[(r + 3) * TL_P + c4]);
            const unsigned C = row[0];
            const unsigned Rt = __byte_perm(row[0], row[1], 0x6543), Lf = __byte_perm(row[-1], row[0], 0x4321);   // x+3, x-3
            const unsigned Dn = row[3 * (TL_P / 4)], Up = row[-3 * (TL_P / 4)];                                   // y+3 (k=0), y-3 (k=8)
            // A_k: centre brighter than ring_k by more than th; B_k: darker
            const unsigned A0 = __vcmpgtu4(__vsubus4(C, Dn), T4), A8 = __vcmpgtu4(__vsubus4(C, Up), T4);
            const unsigned A4 = __vcmpgtu4(__vsubus4(C, Rt), T4), A12 = __vcmpgtu4(__vsubus4(C, Lf), T4);
            const unsigned B0 = __vcmpgtu4(__vsubus4(Dn, C), T4), B8 = __vcmpgtu4(__vsubus4(Up, C), T4);
            const unsigned B4 = __vcmpgtu4(__vsubus4(Rt, C), T4), B12 = __vcmpgtu4(__vsubus4(Lf, C), T4);
            pm = (((A0 | A8) & (A4 | A12)) | ((B0 | B8) & (B4 | B12))) & 0x01010101u;
            if (c4 < xo) pm &= ~0u << (8 * (xo - c4));                                    // clip the first and the last group of a row
            if (c4 + 4 > xo + aw) pm &= (1u << (8 * (xo + aw - c4))) - 1u;
        }
        // warp prefix of the 0..4 survivors per lane from three ballots (the order inside the queue does not matter)
        const int cnt = __popc(pm);
        const unsigned b0 = __ballot_sync(0xffffffffu, cnt & 1), b1 = __ballot_sync(0xffffffffu, cnt & 2), b2 = __ballot_sync(0xffffffffu, cnt & 4);
        const int tot = __popc(b0) + 2 * __popc(b1) + 4 * __popc(b2);
        int base = 0;
        if (lane == 0 && tot) base = atomicAdd(&s_qn, tot);
        base = __shfl_sync(0xffffffffu, base, 0) + __popc(b0 & ltmask) + 2 * __popc(b1 & ltmask) + 4 * __popc(b2 & ltmask);
        const int p0 = (r << 6) + c4 - xo;
#pragma unroll
        for (int k = 0; k < 4; k++) if (pm & (1u << (8 * k))) s_q[base++] = (unsigned short)(p0 + k);
    }
    __syncthreads();
    // phase B1: the exact corner test (9 contiguous ring pixels all brighter or all darker by more than th <=> score >= th) for the queued
    // pixels, on 16-bit arc masks built with byte-SIMD compares; corners are compacted IN PLACE (entries are read a block of 128 ahead of
    // where the survivors are written)
    const int nq = s_qn;
    for (int qb = 0; qb < nq; qb += 128) {
        const int qi = qb + tid;
        bool corner = false;
        int p = 0;
        if (qi < nq) {
            p = s_q[qi];
            const uint8_t* P = &s_img[((p >> 6) + 3) * TL_P + (p & 63) + xo];
            const unsigned v = P[0];
            const unsigned LO4 = 0x01010101u * (unsigned)max((int)v - th, 0), HI4 = 0x01010101u * (unsigned)min((int)v + th, 255);
            const unsigned W0 = P[3 * TL_P] | (P[3 * TL_P + 1] << 8) | (P[2 * TL_P + 2] << 16) | (P[TL_P + 3] << 24);                    // ring 0..3
            const unsigned W1 = P[3] | (P[-TL_P + 3] << 8) | (P[-2 * TL_P + 2] << 16) | (P[-3 * TL_P + 1] << 24);                       // 4..7
            const unsigned W2 = P[-3 * TL_P] | (P[-3 * TL_P - 1] << 8) | (P[-2 * TL_P - 2] << 16) | (P[-TL_P - 3] << 24);               // 8..11
            const unsigned W3 = P[-3] | (P[TL_P - 3] << 8) | (P[2 * TL_P - 2] << 16) | (P[3 * TL_P - 1] << 24);                         // 12..15
            // byte masks -> 4 bits each: (m & 0x08040201) * 0x01010101 >> 24
#define SSLPL_NIB(m) ((((m) & 0x08040201u) * 0x01010101u) >> 24)
            const unsigned br = SSLPL_NIB(__vcmpltu4(W0, LO4)) | (SSLPL_NIB(__vcmpltu4(W1, LO4)) << 4) | (SSLPL_NIB(__vcmpltu4(W2, LO4)) << 8) | (SSLPL_NIB(__vcmpltu4(W3, LO4)) << 12);
            const unsigned dk = SSLPL_NIB(__vcmpgtu4(W0, HI4)) | (SSLPL_NIB(__vcmpgtu4(W1, HI4)) << 4) | (SSLPL_NIB(__vcmpgtu4(W2, HI4)) << 8) | (SSLPL_NIB(__vcmpgtu4(W3, HI4)) << 12);
#undef SSLPL_NIB
            unsigned xb = br | (br << 16), xd = dk | (dk << 16);                          // the ring twice: runs may wrap
            unsigned ab = xb & (xb >> 1), ad = xd & (xd >> 1);
            ab &= ab >> 2; ad &= ad >> 2;
            ab &= ab >> 4; ad &= ad >> 4;
            ab &= xb >> 8; ad &= xd >> 8;                                                 // bit k: ring k..k+8 all set
            corner = ((ab | ad) & 0xffffu) != 0u;
        }
        const unsigned cb = __ballot_sync(0xffffffffu, corner);
        __syncthreads();                                                                 // every entry of this block has been read
        int base = 0;
        if (lane == 0 && cb) base = atomicAdd(&s_qc, __popc(cb));
        base = __shfl_sync(0xffffffffu, base, 0) + __popc(cb & ltmask);
        if (corner) s_q[base] = (unsigned short)p;
    }
    __syncthreads();
    // phase B2: the score of the corners, all lanes busy
    const int nc = s_qc;
    for (int qi = tid; qi < nc; qi += 128) {
        const int p = s_q[qi], r = p >> 6, c = p & 63;
        s_sc[(r + 1) * FAST_TP + c + 1] = (uint8_t)fast_score_tile(&s_img[(r + 3) * TL_P + c + xo], TL_P, th);
    }
    __syncthreads();
    // in-cell NMS of the corners; survivors as one bit per pixel in a 64-bit mask per row (all, and those >= iniTh)
    for (int qi = tid; qi < nc; qi += 128) {
        const int p = s_q[qi], y = p >> 6, x = p & 63;
        const uint8_t* c = &s_sc[(y + 1) * FAST_TP + x + 1];
        const int sc = c[0];
        if (sc > c[-1] && sc > c[1] && sc > c[-FAST_TP - 1] && sc > c[-FAST_TP] && sc > c[-FAST_TP + 1] &&
            sc > c[FAST_TP - 1] && sc > c[FAST_TP] && sc > c[FAST_TP + 1]) {
            atomicOr(&s_rowall[y], 1ull << x);
            if (sc >= g.iniTh) atomicOr(&s_rowhi[y], 1ull << x);
        }
    }
    __syncthreads();
    const unsigned long long mh = tid < ah ? s_rowhi[tid] : 0ull;
    const int any_hi = __syncthreads_or(mh != 0ull);
    unsigned long long m = tid < ah ? (any_hi ? mh : s_rowall[tid]) : 0ull;             // thread = row: raster order by an exclusive scan over the rows
    int total;
    int off = block_exclusive_scan(__popcll(m), s_warp, &total);
    uint32_t* out = ws.cand + (long long)f * g.cand_stride + L.cand_off + (long long)ci * L.cell_cap;
    const int ox = iniX + 3 - MINB, oy = iniY + 3 - MINB;   // coordinates relative to (minBorderX, minBorderY)
    for (; m; m &= m - 1ull) {
        const int x = __ffsll((long long)m) - 1;
        const int sc = s_sc[(tid + 1) * FAST_TP + x + 1];
        if (off < L.cell_cap) out[off] = (uint32_t)(x + ox) | ((uint32_t)(tid + oy) << 12) | ((uint32_t)sc << 24);
        off++;
    }
    if (tid == 0) { *cnt_out = min(total, L.cell_cap); if (total > L.cell_cap) atomicOr(ws.err, DERR_KEY_OVERFLOW); }
}

// ------------------------------------------------------------------------------------------------
// DistributeOctTree in array form (validated against the list form of the oracle):
//   * list order == descending pool index (roots stored reversed, every push_front appends to the pool)
//   * keys of a node are always in ascending candidate order, so only key->node is stored
//   * careful-phase sort key (size, creation counter) == (count, pool index)
// ------------------------------------------------------------------------------------------------
struct Oct {
    uint32_t* kxyr; int* knode; short4* nbox; int* ncnt; int* nq; uint8_t* nalive; unsigned* nbest; int* scan; int* ord;
    int C, N, pool_cap;
};

__device__ __forceinline__ int oct_quadrant(const short4 b, uint32_t xyr) {
    const int x = xyr & 0xfff, y = (xyr >> 12) & 0xfff;
    const int mx = b.x + ((b.z - b.x + 1) >> 1), my = b.y + ((b.w - b.y + 1) >> 1);   // ceil(d/2.f), ORBextractor.cc:483-484
    return x < mx ? (y < my ? 0 : 2) : (y < my ? 1 : 3);
}

// Divide the nodes ord[0..ne) in that order (children appended n1..n4); with limitN >= 0 stop after the
// first division that brings the list size to >= limitN (ORBextractor.cc:730).  Block-wide; returns false on overflow.
__device__ bool oct_divide(const Oct& o, int ne, int limitN, int* s_warp, int* s_size, int* s_top, int* s_pass0, int* s_pass1,
                           int* s_nexp, int* s_tmp, int* err) {
    const int tid = threadIdx.x, T = blockDim.x;
    for (int j = tid; j < ne; j += T) {
        int nd = o.ord[j];
        o.nq[4 * nd] = 0; o.nq[4 * nd + 1] = 0; o.nq[4 * nd + 2] = 0; o.nq[4 * nd + 3] = 0;
        o.nalive[nd] = 2;
    }
    if (tid == 0) { *s_tmp = ne; *s_nexp = 0; }
    __syncthreads();
    for (int k = tid; k < o.C; k += T) {
        int nd = o.knode[k];
        if (o.nalive[nd] == 2) atomicAdd(&o.nq[4 * nd + oct_quadrant(o.nbox[nd], o.kxyr[k])], 1);
    }
    __syncthreads();
    int commit = ne;
    if (limitN >= 0) {
        for (int j = tid; j < ne; j += T) {
            const int* q = &o.nq[4 * o.ord[j]];
            o.scan[j] = (q[0] > 0) + (q[1] > 0) + (q[2] > 0) + (q[3] > 0) - 1;
        }
        __syncthreads();
        block_scan_array(o.scan, ne, s_warp);
        const int size = *s_size;
        for (int j = tid; j < ne; j += T) {
            const int* q = &o.nq[4 * o.ord[j]];
            int g = (q[0] > 0) + (q[1] > 0) + (q[2] > 0) + (q[3] > 0) - 1;
            if (size + o.scan[j] + g >= limitN) atomicMin(s_tmp, j + 1);
        }
        __syncthreads();
        commit = *s_tmp;
    }
    for (int j = tid; j < commit; j += T) {
        const int* q = &o.nq[4 * o.ord[j]];
        o.scan[j] = (q[0] > 0) + (q[1] > 0) + (q[2] > 0) + (q[3] > 0);
    }
    __syncthreads();
    const int created = block_scan_array(o.scan, commit, s_warp);
    const int top = *s_top;
    if (top + created > o.pool_cap) { if (tid == 0) atomicOr(err, DERR_POOL_OVERFLOW); return false; }
    for (int j = tid; j < ne; j += T) {
        const int nd = o.ord[j];
        if (j >= commit) { o.nalive[nd] = 1; continue; }
        const short4 b = o.nbox[nd];
        const short mx = b.x + ((b.z - b.x + 1) >> 1), my = b.y + ((b.w - b.y + 1) >> 1);
        int idx = top + o.scan[j];
#pragma unroll
        for (int c = 0; c < 4; c++) {
            const int cnt = o.nq[4 * nd + c];
            if (cnt > 0) {
                short4 cb;
                cb.x = (c & 1) ? mx : b.x; cb.z = (c & 1) ? b.z : mx;
                cb.y = (c & 2) ? my : b.y; cb.w = (c & 2) ? b.w : my;
                o.nbox[idx] = cb; o.ncnt[idx] = cnt; o.nalive[idx] = 1;
                o.nq[4 * nd + c] = idx;
                if (cnt > 1) atomicAdd(s_nexp, 1);
                idx++;
            }
        }
        o.nalive[nd] = 3;
    }
    __syncthreads();
    for (int k = tid; k < o.C; k += T) {
        int nd = o.knode[k];
        if (o.nalive[nd] == 3) o.knode[k] = o.nq[4 * nd + oct_quadrant(o.nbox[nd], o.kxyr[k])];
    }
    __syncthreads();
    for (int j = tid; j < commit; j += T) o.nalive[o.ord[j]] = 0;
    if (tid == 0) { *s_size += created - commit; *s_pass0 = top; *s_pass1 = top + created; *s_top = top + created; }
    __syncthreads();
    return true;
}

__global__ void __launch_bounds__(256) k_octree(const __grid_constant__ OrbGeom g, OrbWs ws) {
    extern __shared__ unsigned long long s_keys[];
    __shared__ int s_warp[33];
    __shared__ int s_size, s_top, s_pass0, s_pass1, s_nexp, s_tmp, s_ne;
    const int l = blockIdx.x, f = blockIdx.y, tid = threadIdx.x, T = blockDim.x;
    const LevelGeom& L = g.lv[l];
    int* lvl_cnt = ws.lvl_cnt + f * MAXL + l;
    Oct o;
    o.kxyr = ws.kxyr + (long long)f * g.key_stride + L.key_off;
    o.knode = ws.knode + (long long)f * g.key_stride + L.key_off;
    const long long po = (long long)f * g.pool_stride + L.pool_off;
    o.nbox = ws.nbox + po; o.ncnt = ws.ncnt + po; o.nq = ws.nq + 4 * po; o.nalive = ws.nalive + po;
    o.nbest = ws.nbest + po; o.scan = ws.scan + po; o.ord = ws.ord + po;
    o.N = L.nfeat; o.pool_cap = L.pool_cap;
    // --- gather the per-cell candidate lists into vToDistributeKeys order (cell rows, cell cols, raster)
    const int* cell_cnt = ws.cell_cnt + (long long)f * g.total_cells + L.cell_base;
    int* cell_off = ws.cell_off + (long long)f * g.total_cells + L.cell_base;
    for (int c = tid; c < L.ncells; c += T) cell_off[c] = cell_cnt[c];
    __syncthreads();
    const int C = block_scan_array(cell_off, L.ncells, s_warp);
    o.C = C;
    if (C > L.key_cap) { if (tid == 0) { atomicOr(ws.err, DERR_KEY_OVERFLOW); *lvl_cnt = 0; } return; }
    {
        const uint32_t* cand = ws.cand + (long long)f * g.cand_stride + L.cand_off;
        const int lane = tid & 31, wid = tid >> 5, nw = T >> 5;
        for (int c = wid; c < L.ncells; c += nw) {
            const int n = cell_cnt[c], off = cell_off[c];
            for (int s = lane; s < n; s += 32) o.kxyr[off + s] = cand[(long long)c * L.cell_cap + s];
        }
    }
    __syncthreads();
    const int dx = L.maxBX - MINB, dy = L.maxBY - MINB;
    const int nIni = (int)roundf(__fdiv_rn((float)dx, (float)dy));                      // ORBextractor.cc:542
    if (C == 0 || nIni <= 0 || nIni > o.pool_cap) { if (tid == 0) *lvl_cnt = 0; return; }
    const float hX = __fdiv_rn((float)dx, (float)nIni);                                  // :544
    for (int i = tid; i < nIni; i += T) {
        const int idx = nIni - 1 - i;
        short4 b;
        b.x = (short)(int)__fmul_rn(hX, (float)i); b.z = (short)(int)__fmul_rn(hX, (float)(i + 1)); b.y = 0; b.w = (short)dy;
        o.nbox[idx] = b; o.ncnt[idx] = 0; o.nalive[idx] = 1;
    }
    __syncthreads();
    for (int k = tid; k < C; k += T) {
        int r = (int)__fdiv_rn((float)(o.kxyr[k] & 0xfff), hX);                         // :569
        r = min(r, nIni - 1);
        o.knode[k] = nIni - 1 - r;
        atomicAdd(&o.ncnt[nIni - 1 - r], 1);
    }
    __syncthreads();
    if (tid == 0) {
        int size = 0;
        for (int i = 0; i < nIni; i++) { if (o.ncnt[i] == 0) o.nalive[i] = 0; else size++; }
        s_size = size; s_pass0 = 0; s_pass1 = nIni; s_top = nIni;
    }
    __syncthreads();
    const int N = o.N;
    bool ok = true;
    while (true) {                                                                        // :591
        const int prevSize = s_size, p0 = s_pass0, p1 = s_pass1, m = p1 - p0;
        for (int r = tid; r < m; r += T) { int nd = p1 - 1 - r; o.scan[r] = (o.nalive[nd] == 1 && o.ncnt[nd] > 1); }
        __syncthreads();
        const int ne = block_scan_array(o.scan, m, s_warp);
        for (int r = tid; r < m; r += T) { int nd = p1 - 1 - r; if (o.nalive[nd] == 1 && o.ncnt[nd] > 1) o.ord[o.scan[r]] = nd; }
        __syncthreads();
        ok = oct_divide(o, ne, -1, s_warp, &s_size, &s_top, &s_pass0, &s_pass1, &s_nexp, &s_tmp, ws.err);
        if (!ok) break;
        const int size = s_size, nToExpand = s_nexp;
        if (size >= N || size == prevSize) break;                                         // :669
        if (size + nToExpand * 3 > N) {                                                   // :673
            while (true) {
                const int prev2 = s_size, q0 = s_pass0, q1 = s_pass1;
                if (tid == 0) s_ne = 0;
                __syncthreads();
                for (int nd = q0 + tid; nd < q1; nd += T)
                    if (o.nalive[nd] == 1 && o.ncnt[nd] > 1) {
                        int slot = atomicAdd(&s_ne, 1);
                        if (slot < g.sort_cap) s_keys[slot] = ((unsigned long long)o.ncnt[nd] << 32) | (unsigned)nd;
                    }
                __syncthreads();
                const int ne2 = s_ne;
                if (ne2 > g.sort_cap) { if (tid == 0) atomicOr(ws.err, DERR_SORT_OVERFLOW); ok = false; break; }
                int P = 1; while (P < ne2) P <<= 1;
                for (int i = ne2 + tid; i < P; i += T) s_keys[i] = 0ull;
                __syncthreads();
                for (int k = 2; k <= P; k <<= 1)                                          // bitonic sort, descending (:684-685)
                    for (int j = k >> 1; j > 0; j >>= 1) {
                        for (int i = tid; i < P; i += T) {
                            const int ixj = i ^ j;
                            if (ixj > i) {
                                const unsigned long long a = s_keys[i], b = s_keys[ixj];
                                const bool desc = (i & k) == 0;
                                if (desc ? (a < b) : (a > b)) { s_keys[i] = b; s_keys[ixj] = a; }
                            }
                        }
                        __syncthreads();
                    }
                for (int j = tid; j < ne2; j += T) o.ord[j] = (int)(s_keys[j] & 0xffffffffull);
                __syncthreads();
                ok = oct_divide(o, ne2, N, s_warp, &s_size, &s_top, &s_pass0, &s_pass1, &s_nexp, &s_tmp, ws.err);
                if (!ok) break;
                if (s_size >= N || s_size == prev2) break;                                // :734
            }
            break;
        }
    }
    if (!ok) { if (tid == 0) *lvl_cnt = 0; return; }
    // --- retain the best keypoint of every node (max response, first wins), in list order      :741-760
    const int top = s_top;
    for (int nd = tid; nd < top; nd += T) o.nbest[nd] = 0u;
    __syncthreads();
    for (int k = tid; k < C; k += T) atomicMax(&o.nbest[o.knode[k]], ((o.kxyr[k] >> 24) << 24) | (0xFFFFFFu - (unsigned)k));
    for (int r = tid; r < top; r += T) o.scan[r] = (o.nalive[top - 1 - r] == 1);
    __syncthreads();
    const int total = block_scan_array(o.scan, top, s_warp);
    uint32_t* out = ws.lvl_kp + (long long)f * g.kp_total_cap + L.kp_base;
    for (int r = tid; r < top; r += T) {
        const int nd = top - 1 - r;
        if (o.nalive[nd] == 1) {
            const int pos = o.scan[r];
            if (pos < L.kp_cap) {
                const uint32_t xyr = o.kxyr[0xFFFFFFu - (o.nbest[nd] & 0xFFFFFFu)];
                out[pos] = ((xyr & 0xfff) + MINB) | ((((xyr >> 12) & 0xfff) + MINB) << 12) | (xyr & 0xff000000u);
            }
        }
    }
    if (tid == 0) { *lvl_cnt = min(total, L.kp_cap); if (total > L.kp_cap) atomicOr(ws.err, DERR_KP_OVERFLOW); }
}

// ------------------------------------------------------------------------------------------------
// GaussianBlur 7x7 sigma 2, OpenCV 4.13 fixed-point path (SURVEY.md A.2), BORDER_REFLECT_101
// ------------------------------------------------------------------------------------------------
template <bool TMA>
__global__ void __launch_bounds__(256) k_blur(const __grid_constant__ OrbGeom g, OrbWs ws, View v, const CUtensorMap* tm) {
    __shared__ __align__(128) uint8_t s_img[TL_IH * TL_P];
    __shared__ __align__(16) unsigned s_pair[TL_IH * TL_W];             // [r][x] = row pass of row r | row r+1 << 16
    __shared__ __align__(8) uint64_t s_bar;
    const int tile = blockIdx.x, f = blockIdx.y, tid = threadIdx.x;
    int l = 0;
    while (l + 1 < g.nlevels && tile >= g.lv[l + 1].tile_base) l++;
    const LevelGeom& L = g.lv[l];
    const int t = tile - L.tile_base, ty = t / L.tiles_x, tx = t - ty * L.tiles_x;
    const int x0 = tx * TL_W, y0 = ty * TL_H, bx = x0 - TL_X, by = y0 - 3;
    int pitch;
    const uint8_t* img = level_ptr(g, ws, v, l, f, &pitch);
    const bool interior = bx >= 0 && by >= 0 && x0 + TL_W + 3 <= L.w && y0 + TL_H + 3 <= L.h;
    if (TMA || interior) {
        stage_box<TMA>(s_img, &s_bar, tm, img, pitch, L.w, L.h, l, f, bx, by);
        if (!interior) {
            // BORDER_REFLECT_101 on top of the zero-filled box: columns first (valid rows), then whole rows
            for (int i = tid; i < TL_IH * 8; i += 256) {
                const int r = i >> 3, k = i & 7, gy = by + r;
                if (gy < 0 || gy >= L.h) continue;
                const int c = k < 4 ? TL_X - 4 + k : (k - 4) + (L.w - bx);   // left halo cols (gx = x0-4..x0-1), right cols gx = w..w+3
                const int gx = bx + c;
                if (c >= 0 && c < TL_P && (gx < 0 || gx >= L.w)) { const int sxx = reflect101(gx, L.w) - bx; if (sxx >= 0 && sxx < TL_P) s_img[r * TL_P + c] = s_img[r * TL_P + sxx]; }
            }
            __syncthreads();
            for (int i = tid; i < 6 * TL_P; i += 256) {
                const int k = i / TL_P, c = i - k * TL_P;
                const int r = k < 3 ? k : (k - 3) + (L.h - by);            // top halo rows 0..2, bottom rows h-by..h-by+2
                const int gy = by + r;
                if (r >= 0 && r < TL_IH && (gy < 0 || gy >= L.h)) { const int sr = reflect101(gy, L.h) - by; if (sr >= 0 && sr < TL_IH) s_img[r * TL_P + c] = s_img[sr * TL_P + c]; }
            }
            __syncthreads();
        }
    } else {
        for (int i = tid; i < TL_IH * (TL_W + 6); i += 256) {
            const int r = i / (TL_W + 6), c = i - r * (TL_W + 6) + TL_X - 3;
            s_img[r * TL_P + c] = __ldg(img + (long long)reflect101(by + r, L.h) * pitch + reflect101(bx + c, L.w));
        }
        __syncthreads();
    }
    // Packed arithmetic (taps 18 34 48 56 48 34 18): horizontal pass = two dp4a per output on byte windows cut out of three
    // aligned words with funnel shifts (TL_X - 3 = 13 = 12 + 1); the u16 results are stored as vertical PAIRS
    // (row r | row r+1 << 16) so that the vertical pass is four dp2a per output.  Partial sums stay below 2^16 / 2^32: exact.
    static_assert(TL_X == 16 && TL_P % 4 == 0, "word-aligned row reads assume TL_X == 16");
    constexpr unsigned T0 = 18u | (34u << 8) | (48u << 16) | (56u << 24), T1 = 48u | (34u << 8) | (18u << 16);
    unsigned short* s_half = reinterpret_cast<unsigned short*>(s_pair);
    for (int i = tid; i < TL_IH * (TL_W / 4); i += 256) {
        const int r = i >> 4, x4 = (i & 15) * 4;
        const unsigned* w = reinterpret_cast<const unsigned*>(&s_img[r * TL_P + x4 + TL_X - 4]);
        const unsigned w0 = w[0], w1 = w[1], w2 = w[2];                   // output k uses bytes 1 + k .. 7 + k of this window
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const unsigned A = (k < 3) ? __funnelshift_r(w0, w1, 8 * (k + 1)) : w1;
            const unsigned B = (k < 3) ? __funnelshift_r(w1, w2, 8 * (k + 1)) : w2;
            const unsigned q = __dp4a(A, T0, __dp4a(B, T1, 0u));          // <= 65280
            s_half[(r * TL_W + x4 + k) * 2] = (unsigned short)q;
            if (r > 0) s_half[((r - 1) * TL_W + x4 + k) * 2 + 1] = (unsigned short)q;
        }
    }
    __syncthreads();
    uint8_t* out = ws.blur + (long long)f * g.blur_stride + L.blur_off;
    constexpr unsigned C01 = 18u | (34u << 8), C23 = 48u | (56u << 8), C45 = 48u | (34u << 8), C6 = 18u;
    for (int i = tid; i < TL_H * (TL_W / 4); i += 256) {
        const int yy = i >> 4, x4 = (i & 15) * 4;
        if (y0 + yy >= L.h || x0 + x4 >= L.w) continue;
        const uint4 p0 = *reinterpret_cast<const uint4*>(&s_pair[yy * TL_W + x4]), p2 = *reinterpret_cast<const uint4*>(&s_pair[(yy + 2) * TL_W + x4]);
        const uint4 p4 = *reinterpret_cast<const uint4*>(&s_pair[(yy + 4) * TL_W + x4]), p6 = *reinterpret_cast<const uint4*>(&s_pair[(yy + 6) * TL_W + x4]);
        const unsigned a0 = __dp2a_lo(p0.x, C01, __dp2a_lo(p2.x, C23, __dp2a_lo(p4.x, C45, __dp2a_lo(p6.x, C6, 32768u))));
        const unsigned a1 = __dp2a_lo(p0.y, C01, __dp2a_lo(p2.y, C23, __dp2a_lo(p4.y, C45, __dp2a_lo(p6.y, C6, 32768u))));
        const unsigned a2 = __dp2a_lo(p0.z, C01, __dp2a_lo(p2.z, C23, __dp2a_lo(p4.z, C45, __dp2a_lo(p6.z, C6, 32768u))));
        const unsigned a3 = __dp2a_lo(p0.w, C01, __dp2a_lo(p2.w, C23, __dp2a_lo(p4.w, C45, __dp2a_lo(p6.w, C6, 32768u))));
        const uint32_t o4 = (a0 >> 16) | ((a1 >> 16) << 8) | ((a2 >> 16) << 16) | ((a3 >> 16) << 24);
        *reinterpret_cast<uint32_t*>(out + (long long)(y0 + yy) * L.bpitch + x0 + x4) = o4;      // bytes past w are padding
    }
}

// ------------------------------------------------------------------------------------------------
// IC_Angle + rBRIEF + KeyPoint assembly: one warp per output keypoint
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_orient_desc(const __grid_constant__ OrbGeom g, OrbWs ws, View v) {
    __shared__ signed char s_pat[1024];
    for (int i = threadIdx.x; i < 1024; i += 256) s_pat[i] = c_pattern[i];
    __syncthreads();
    const int lane = threadIdx.x & 31, slot = blockIdx.x * 8 + (threadIdx.x >> 5), f = blockIdx.y;
    const int* lc = ws.lvl_cnt + f * MAXL;
    int l = -1, pref = 0, total = 0;
    for (int i = 0; i < g.nlevels; i++) {
        const int c = lc[i];
        if (l < 0 && slot < total + c) { l = i; pref = total; }
        total += c;
    }
    if (slot == 0 && lane == 0) ws.nkp[f] = total;
    if (l < 0) return;
    const LevelGeom& L = g.lv[l];
    const uint32_t xyr = ws.lvl_kp[(long long)f * g.kp_total_cap + L.kp_base + (slot - pref)];
    const int x = xyr & 0xfff, y = (xyr >> 12) & 0xfff, resp = xyr >> 24;
    int pitch;
    const uint8_t* center = level_ptr(g, ws, v, l, f, &pitch);
    center += (long long)y * pitch + x;
    // IC_Angle (ORBextractor.cc:77-104): m10 = sum u*I, m01 = sum v*I over the 31-px disc (exact integers)
    int m10 = 0, m01 = 0;
    const int u = lane - HALF_PATCH;
    if (lane < 31) {
#pragma unroll
        for (int vv = -HALF_PATCH; vv <= HALF_PATCH; vv++) {
            if (abs(u) <= g.umax[abs(vv)]) {
                const int val = __ldg(center + (long long)vv * pitch + u);
                m10 += u * val; m01 += vv * val;
            }
        }
    }
    m10 = __reduce_add_sync(0xffffffffu, m10);
    m01 = __reduce_add_sync(0xffffffffu, m01);
    const float angle = fast_atan2_deg((float)m01, (float)m10);
    // computeOrbDescriptor (ORBextractor.cc:107-147); lane i produces byte i
    const float factorPI = (float)(3.141592653589793238462643383279502884 / 180.0);   // == (float)(CV_PI/180.f)
    const float rad = __fmul_rn(angle, factorPI);
    const float a = (float)cos((double)rad), b = (float)sin((double)rad);
    const uint8_t* bc = ws.blur + (long long)f * g.blur_stride + L.blur_off + (long long)y * L.bpitch + x;
    const signed char* pat = s_pat + lane * 32;
    int val = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const float px0 = (float)pat[4 * k], py0 = (float)pat[4 * k + 1], px1 = (float)pat[4 * k + 2], py1 = (float)pat[4 * k + 3];
        const int r0 = __float2int_rn(__fadd_rn(__fmul_rn(px0, b), __fmul_rn(py0, a)));
        const int c0 = __float2int_rn(__fsub_rn(__fmul_rn(px0, a), __fmul_rn(py0, b)));
        const int r1 = __float2int_rn(__fadd_rn(__fmul_rn(px1, b), __fmul_rn(py1, a)));
        const int c1 = __float2int_rn(__fsub_rn(__fmul_rn(px1, a), __fmul_rn(py1, b)));
        const int t0 = __ldg(bc + (long long)r0 * L.bpitch + c0), t1 = __ldg(bc + (long long)r1 * L.bpitch + c1);
        val |= (t0 < t1) << k;
    }
    // 32 descriptor bytes -> two coalesced 16-byte stores (lanes 0 and 4 of each octet hold the words)
    uint32_t w = (uint32_t)val << (8 * (lane & 3));
    w |= __shfl_xor_sync(0xffffffffu, w, 1);
    w |= __shfl_xor_sync(0xffffffffu, w, 2);
    const uint32_t w0 = __shfl_sync(0xffffffffu, w, (lane & 16) + 0), w1 = __shfl_sync(0xffffffffu, w, (lane & 16) + 4),
                   w2 = __shfl_sync(0xffffffffu, w, (lane & 16) + 8), w3 = __shfl_sync(0xffffffffu, w, (lane & 16) + 12);
    const long long oidx = (long long)f * g.kp_total_cap + slot;
    if ((lane & 15) == 0) reinterpret_cast<uint4*>(ws.desc + oidx * 32)[lane >> 4] = make_uint4(w0, w1, w2, w3);
    if (lane < 7) {                                                              // cv::KeyPoint, 7 words
        float fx = (float)x, fy = (float)y;
        if (l != 0) { fx = __fmul_rn(fx, L.scale); fy = __fmul_rn(fy, L.scale); }     // ORBextractor.cc:1096-1100
        float wv;
        switch (lane) {
            case 0: wv = fx; break;
            case 1: wv = fy; break;
            case 2: wv = L.patch_size; break;
            case 3: wv = angle; break;
            case 4: wv = (float)resp; break;
            case 5: wv = __int_as_float(l); break;
            default: wv = __int_as_float(-1); break;
        }
        reinterpret_cast<float*>(ws.kps + oidx)[lane] = wv;
    }
}

}  // namespace sslpl

// =================================================================================================
// Host side of the handle
// =================================================================================================
using namespace sslpl;

struct sslpl_orb {
    sslpl_orb_params p;
    std::vector<float> scale, invscale, sigma2, invsigma2;
    std::vector<int> nfeat, umax;
    cudaStream_t stream = nullptr, own_stream = nullptr;
    uint8_t* arena = nullptr; size_t arena_size = 0;
    OrbGeom g; OrbWs ws; View view;
    uint8_t* d_input = nullptr;         // staging for host frames
    int cur_w = 0, cur_h = 0, cur_frames = 0;
    long long launches = 0;
    bool profiling = false;
    std::vector<cudaEvent_t> ev; std::vector<const char*> ev_name; int ev_n = 0;
    int* h_err = nullptr;               // pinned
    int octree_smem = 0;
    CUtensorMap tm[MAXL];               // per pyramid level: 3-D (x, y, frame) u8 tensor map with the 96x38 box of the stencil kernels
                                        // (level 0 re-encoded per call: the input view moves)
    PFN_cuTensorMapEncodeTiled_v12000 encode = nullptr;
    bool tma_levels_ok = false, use_tma = true;
    const uint8_t* tm0_base = nullptr; int tm0_pitch = 0, tm0_frames = 0; long long tm0_fs = 0;
};

namespace {

inline int cvRoundF(float v) { return (int)lrintf(v); }
inline int cvFloorF(float v) { int i = (int)v; return i - (i > v); }
inline int cvCeilF(float v) { int i = (int)v; return i + (i < v); }

// ORBextractor::ORBextractor, ORBextractor.cc:410-470
void make_tables(sslpl_orb* h) {
    const int L = h->p.nlevels;
    const double sfd = (double)h->p.scaleFactor;          // member `double scaleFactor`, ORBextractor.h:96
    h->scale.assign(L, 1.f); h->sigma2.assign(L, 1.f); h->invscale.assign(L, 1.f); h->invsigma2.assign(L, 1.f);
    for (int i = 1; i < L; i++) { h->scale[i] = (float)(h->scale[i - 1] * sfd); h->sigma2[i] = h->scale[i] * h->scale[i]; }
    for (int i = 0; i < L; i++) { h->invscale[i] = 1.0f / h->scale[i]; h->invsigma2[i] = 1.0f / h->sigma2[i]; }
    h->nfeat.assign(L, 0);
    float factor = (float)(1.0f / sfd);
    float nDesired = h->p.nfeatures * (1 - factor) / (1 - (float)pow((double)factor, (double)L));
    int sum = 0;
    for (int l = 0; l < L - 1; l++) { h->nfeat[l] = cvRoundF(nDesired); sum += h->nfeat[l]; nDesired *= factor; }
    h->nfeat[L - 1] = std::max(h->p.nfeatures - sum, 0);
    h->umax.assign(HALF_PATCH + 1, 0);
    int v, v0, vmax = cvFloorF(HALF_PATCH * sqrtf(2.f) / 2 + 1), vmin = cvCeilF(HALF_PATCH * sqrtf(2.f) / 2);
    const double hp2 = HALF_PATCH * HALF_PATCH;
    for (v = 0; v <= vmax; ++v) h->umax[v] = (int)lrint(sqrt(hp2 - v * v));
    for (v = HALF_PATCH, v0 = 0; v >= vmin; --v) { while (h->umax[v0] == h->umax[v0 + 1]) ++v0; h->umax[v] = v0; ++v0; }
}

// Geometry for a frame size; with alloc==nullptr only sizes are computed.
void make_geometry(const sslpl_orb* h, int W, int H, OrbGeom& g, std::vector<int2>* rtab) {
    memset(&g, 0, sizeof(g));
    const int L = h->p.nlevels;
    g.nlevels = L; g.iniTh = h->p.iniThFAST; g.minTh = h->p.minThFAST;
    for (int i = 0; i < 16; i++) g.umax[i] = h->umax[i];
    long long pyr = 0, blur = 0, cand = 0, key = 0, pool = 0;
    int cells = 0, tiles = 0, kpc = 0, rt = 0, maxN = 2;
    for (int l = 0; l < L; l++) {
        LevelGeom& G = g.lv[l];
        G.w = cvRoundF((float)W * h->invscale[l]); G.h = cvRoundF((float)H * h->invscale[l]);     // ORBextractor.cc:1111-1112
        G.pitch = (int)align_up(G.w, 64);
        G.img_off = pyr; if (l > 0) pyr += align_up((size_t)G.pitch * G.h, 256);
        G.bpitch = (int)align_up(G.w, 64);
        G.blur_off = blur; blur += align_up((size_t)G.bpitch * G.h, 256);
        G.maxBX = G.w - EDGE + 3; G.maxBY = G.h - EDGE + 3;                                          // :777-778
        const float width = (float)(G.maxBX - MINB), height = (float)(G.maxBY - MINB);
        G.nCols = (int)(width / 30.f); G.nRows = (int)(height / 30.f);                             // :786-787
        if (G.nCols > 0 && G.nRows > 0 && width > 0 && height > 0) {
            G.wCell = (int)ceilf(width / G.nCols); G.hCell = (int)ceilf(height / G.nRows);         // :788-789
        } else { G.nCols = G.nRows = 0; G.wCell = G.hCell = 1; }
        G.cell_base = cells; G.ncells = G.nCols * G.nRows; cells += G.ncells;
        G.cell_cap = ((G.wCell + 1) / 2) * ((G.hCell + 1) / 2);        // NMS survivors are pairwise non-adjacent
        G.cand_off = cand; cand += (long long)G.ncells * G.cell_cap;
        G.key_cap = G.ncells * G.cell_cap; G.key_off = key; key += align_up(G.key_cap, 64);
        G.nfeat = h->nfeat[l]; G.kp_cap = G.nfeat + 16; G.kp_base = kpc; kpc += G.kp_cap;
        G.pool_cap = 16 * (G.nfeat + 4) + 64; G.pool_off = pool; pool += align_up(G.pool_cap, 64);
        maxN = std::max(maxN, G.nfeat);
        G.xtab_off = rt; rt += G.w; G.ytab_off = rt; rt += G.h;
        G.tiles_x = (G.w + BLUR_TW - 1) / BLUR_TW; G.tiles_y = (G.h + BLUR_TH - 1) / BLUR_TH;
        G.tile_base = tiles; tiles += G.tiles_x * G.tiles_y;
        G.scale = h->scale[l]; G.patch_size = (float)(int)(31 * h->scale[l]);                      // :836 (int truncation)
    }
    g.total_cells = cells; g.total_tiles = tiles; g.kp_total_cap = kpc;
    g.pyr_stride = pyr; g.blur_stride = blur; g.cand_stride = cand; g.key_stride = key; g.pool_stride = pool;
    int sc = 2; while (sc < maxN) sc <<= 1;
    g.sort_cap = sc;
    if (rtab) {
        rtab->assign(rt, make_int2(0, 0));
        for (int l = 1; l < L; l++) {                                       // cv::resize tables, SURVEY.md A.1
            const LevelGeom& D = g.lv[l]; const LevelGeom& S = g.lv[l - 1];
            for (int axis = 0; axis < 2; axis++) {
                const int dn = axis ? D.h : D.w, sn = axis ? S.h : S.w, off = axis ? D.ytab_off : D.xtab_off;
                const double sc2 = 1.0 / ((double)dn / sn);
                for (int d = 0; d < dn; d++) {
                    float fx = (float)((d + 0.5) * sc2 - 0.5);
                    int sx = cvFloorF(fx); fx -= sx;
                    if (sx < 0) { fx = 0; sx = 0; }
                    if (sx >= sn - 1) { fx = 0; sx = sn - 1; }
                    const int a0 = cvRoundF((1.f - fx) * 2048), a1 = cvRoundF(fx * 2048);
                    (*rtab)[off + d] = make_int2(sx, (a0 & 0xffff) | (a1 << 16));
                }
            }
        }
    }
}

int carve(sslpl_orb* h, Arena& A, const OrbGeom& g, int B, int W, int H) {
    OrbWs& ws = h->ws;
    h->d_input = A.take<uint8_t>((size_t)B * align_up(W, 16) * H + 256);
    ws.pyr = A.take<uint8_t>((size_t)B * g.pyr_stride + 256);
    ws.blur = A.take<uint8_t>((size_t)B * g.blur_stride + 256);
    ws.cand = A.take<uint32_t>((size_t)B * g.cand_stride);
    ws.cell_cnt = A.take<int>((size_t)B * g.total_cells);
    ws.cell_off = A.take<int>((size_t)B * g.total_cells);
    ws.kxyr = A.take<uint32_t>((size_t)B * g.key_stride);
    ws.knode = A.take<int>((size_t)B * g.key_stride);
    ws.nbox = A.take<short4>((size_t)B * g.pool_stride);
    ws.ncnt = A.take<int>((size_t)B * g.pool_stride);
    ws.nq = A.take<int>((size_t)B * g.pool_stride * 4);
    ws.nalive = A.take<uint8_t>((size_t)B * g.pool_stride);
    ws.nbest = A.take<unsigned>((size_t)B * g.pool_stride);
    ws.scan = A.take<int>((size_t)B * g.pool_stride);
    ws.ord = A.take<int>((size_t)B * g.pool_stride);
    ws.lvl_kp = A.take<uint32_t>((size_t)B * g.kp_total_cap);
    ws.lvl_cnt = A.take<int>((size_t)B * MAXL);
    int rt = 0; for (int l = 0; l < g.nlevels; l++) rt += g.lv[l].w + g.lv[l].h;
    ws.rtab = A.take<int2>(rt);
    ws.err = A.take<int>(1);
    ws.kps = A.take<sslpl_keypoint>((size_t)B * g.kp_total_cap);
    ws.desc = A.take<uint8_t>((size_t)B * g.kp_total_cap * 32);
    ws.nkp = A.take<int>(B);
    ws.tmaps = A.take<CUtensorMap>(MAXL);
    return 0;
}

// 3-D u8 tensor map (x, y, frame) with a 96x38x1 box; returns false when the driver entry point is missing or the
// view does not satisfy TMA's 16-byte alignment rules (then the kernels fall back to ordinary loads).
bool encode_level_map(sslpl_orb* h, CUtensorMap* out, const uint8_t* base, int w, int hgt, int pitch, long long frame_stride, int frames) {
    if (!h->encode) return false;
    if ((reinterpret_cast<uintptr_t>(base) & 15) || (pitch & 15) || (frame_stride & 15) || w < 1 || hgt < 1 || frames < 1) return false;
    const cuuint64_t gdim[3] = {(cuuint64_t)w, (cuuint64_t)hgt, (cuuint64_t)frames};
    const cuuint64_t gstr[2] = {(cuuint64_t)pitch, (cuuint64_t)frame_stride};
    const cuuint32_t box[3] = {(cuuint32_t)TL_P, (cuuint32_t)TL_IH, 1u};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    const CUresult r = h->encode(out, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<uint8_t*>(base), gdim, gstr, box, estr,
                                 CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                                 CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

int configure(sslpl_orb* h, int W, int H) {
    if (W == h->cur_w && H == h->cur_h) return SSLPL_OK;
    SSLPL_REQUIRE(W <= h->p.max_width && H <= h->p.max_height, SSLPL_ERR_ARG, "frame larger than the handle's max_width/max_height");
    SSLPL_REQUIRE(W >= 2 * EDGE && H >= 2 * EDGE && W < 4096 && H < 4096, SSLPL_ERR_ARG, "frame size out of range (need 38 <= w,h < 4096)");
    std::vector<int2> rtab;
    make_geometry(h, W, H, h->g, &rtab);
    for (int l = 0; l < h->g.nlevels; l++)
        SSLPL_REQUIRE(h->g.lv[l].w >= 1 && h->g.lv[l].h >= 1, SSLPL_ERR_ARG, "pyramid level collapses to zero size");
    Arena A; A.base = h->arena; A.size = h->arena_size;
    carve(h, A, h->g, h->p.max_batch, W, H);
    SSLPL_REQUIRE(A.used <= h->arena_size, SSLPL_ERR_CAPACITY, "internal: arena too small for this frame size");
    SSLPL_CUDA(cudaStreamSynchronize(h->stream));
    if (!rtab.empty()) SSLPL_CUDA(cudaMemcpy(h->ws.rtab, rtab.data(), rtab.size() * sizeof(int2), cudaMemcpyHostToDevice));
    SSLPL_CUDA(cudaMemset(h->ws.err, 0, sizeof(int)));
    h->octree_smem = h->g.sort_cap * 8;
    SSLPL_CUDA(cudaFuncSetAttribute(k_octree, cudaFuncAttributeMaxDynamicSharedMemorySize, std::max(h->octree_smem, 1024)));
    h->tma_levels_ok = h->encode != nullptr;
    memset(&h->tm, 0, sizeof(h->tm));
    for (int l = 1; l < h->g.nlevels && h->tma_levels_ok; l++)
        h->tma_levels_ok = encode_level_map(h, &h->tm[l], h->ws.pyr + h->g.lv[l].img_off, h->g.lv[l].w, h->g.lv[l].h, h->g.lv[l].pitch,
                                            h->g.pyr_stride, h->p.max_batch);
    if (h->tma_levels_ok) SSLPL_CUDA(cudaMemcpy(h->ws.tmaps, &h->tm, sizeof(h->tm), cudaMemcpyHostToDevice));
    h->tm0_base = nullptr;
    h->cur_w = W; h->cur_h = H;
    return SSLPL_OK;
}

void mark(sslpl_orb* h, const char* name) {
    if (!h->profiling) return;
    if ((int)h->ev.size() <= h->ev_n) { cudaEvent_t e; cudaEventCreate(&e); h->ev.push_back(e); h->ev_name.push_back(name); }
    h->ev_name[h->ev_n] = name;
    cudaEventRecord(h->ev[h->ev_n++], h->stream);
}

// Enqueue the whole extraction for B frames described by `view`.
int run_pipeline(sslpl_orb* h, int B) {
    const OrbGeom& g = h->g;
    cudaStream_t st = h->stream;
    h->ev_n = 0;
    mark(h, "start");
    bool tma = h->use_tma && h->tma_levels_ok;
    if (tma && !(h->tm0_base == h->view.base && h->tm0_pitch == h->view.pitch && h->tm0_fs == h->view.frame_stride && h->tm0_frames >= B)) {
        // level 0 is the caller's buffer: (re-)encode its maps when the view moves
        tma = encode_level_map(h, &h->tm[0], h->view.base, g.lv[0].w, g.lv[0].h, h->view.pitch, h->view.frame_stride, B);
        if (tma) {
            SSLPL_CUDA(cudaMemcpyAsync(h->ws.tmaps, &h->tm[0], sizeof(CUtensorMap), cudaMemcpyHostToDevice, st));
            h->tm0_base = h->view.base; h->tm0_pitch = h->view.pitch; h->tm0_fs = h->view.frame_stride; h->tm0_frames = B;
        } else h->tm0_base = nullptr;
    }
    for (int l = 1; l < g.nlevels; l++) {
        dim3 grid((g.lv[l].w + 127) / 128, (g.lv[l].h + 7) / 8, B), block(32, 8);
        k_resize<<<grid, block, 0, st>>>(g, h->ws, h->view, l);
        h->launches++;
    }
    mark(h, "pyramid");
    if (g.total_cells > 0) {
        if (tma) k_fast<true><<<dim3(g.total_cells, B), 128, 0, st>>>(g, h->ws, h->view, h->ws.tmaps);
        else k_fast<false><<<dim3(g.total_cells, B), 128, 0, st>>>(g, h->ws, h->view, h->ws.tmaps);
        h->launches++;
    }
    mark(h, "fast");
    k_octree<<<dim3(g.nlevels, B), 256, h->octree_smem, st>>>(g, h->ws); h->launches++;
    mark(h, "octree");
    if (tma) k_blur<true><<<dim3(g.total_tiles, B), 256, 0, st>>>(g, h->ws, h->view, h->ws.tmaps);
    else k_blur<false><<<dim3(g.total_tiles, B), 256, 0, st>>>(g, h->ws, h->view, h->ws.tmaps);
    h->launches++;
    mark(h, "blur");
    k_orient_desc<<<dim3((g.kp_total_cap + 7) / 8, B), 256, 0, st>>>(g, h->ws, h->view); h->launches++;
    mark(h, "orient_desc");
    SSLPL_CUDA(cudaGetLastError());
    return SSLPL_OK;
}

int check_device_err(sslpl_orb* h) {
    SSLPL_CUDA(cudaMemcpyAsync(h->h_err, h->ws.err, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    SSLPL_CUDA(cudaStreamSynchronize(h->stream));
    if (*h->h_err) {
        set_error("device-side capacity overflow, flags=0x%x (1 pool, 2 keys, 4 sort, 8 keypoints)", *h->h_err);
        cudaMemsetAsync(h->ws.err, 0, sizeof(int), h->stream);
        return SSLPL_ERR_CAPACITY;
    }
    return SSLPL_OK;
}

}  // namespace

extern "C" {

int sslpl_orb_create(const sslpl_orb_params* p, sslpl_orb** out) {
    SSLPL_REQUIRE(p && out, SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(p->nlevels >= 1 && p->nlevels <= MAXL, SSLPL_ERR_ARG, "nlevels must be in [1,16]");
    SSLPL_REQUIRE(p->nfeatures >= 1 && p->nfeatures <= 200000, SSLPL_ERR_ARG, "nfeatures out of range");
    SSLPL_REQUIRE(p->scaleFactor > 1.0f, SSLPL_ERR_ARG, "scaleFactor must be > 1");
    SSLPL_REQUIRE(p->minThFAST >= 1 && p->iniThFAST >= p->minThFAST && p->iniThFAST < 255, SSLPL_ERR_ARG, "need 1 <= minThFAST <= iniThFAST < 255");
    SSLPL_REQUIRE(p->max_batch >= 1 && p->max_width >= 2 * EDGE && p->max_height >= 2 * EDGE, SSLPL_ERR_ARG, "bad max_batch / max size");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
        set_error("no CUDA device available: libsslpl_b200 has no CPU fallback");
        return SSLPL_ERR_CUDA;
    }
    SSLPL_CUDA(cudaSetDevice(p->device));
    sslpl_orb* h = new sslpl_orb();
    h->p = *p;
    make_tables(h);
    OrbGeom g;
    make_geometry(h, p->max_width, p->max_height, g, nullptr);
    SSLPL_REQUIRE(g.sort_cap * 8 <= 200 * 1024, SSLPL_ERR_UNSUPPORTED, "nfeatures too large for the octree sort buffer");
    Arena A;                                   // dry run for the size
    carve(h, A, g, p->max_batch, p->max_width, p->max_height);
    h->arena_size = A.used + (1 << 20);
    cudaError_t e = cudaMalloc(&h->arena, h->arena_size);
    if (e != cudaSuccess) { set_error("cudaMalloc(%zu) failed: %s", h->arena_size, cudaGetErrorString(e)); delete h; return SSLPL_ERR_CUDA; }
    SSLPL_CUDA(cudaMemset(h->arena, 0, h->arena_size));
    SSLPL_CUDA(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    h->stream = h->own_stream;
    SSLPL_CUDA(cudaHostAlloc((void**)&h->h_err, sizeof(int), cudaHostAllocDefault));
    {   // TMA descriptors are encoded by the driver; resolve the entry point through the runtime (no libcuda link)
        void* fn = nullptr; cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
            h->encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
        else cudaGetLastError();
        const char* e = getenv("SSLPL_NO_TMA");
        h->use_tma = !(e && e[0] == '1');
    }
    *out = h;
    return SSLPL_OK;
}

void sslpl_orb_destroy(sslpl_orb* h) {
    if (!h) return;
    cudaSetDevice(h->p.device);
    // an external stream may already be gone (its owner was destroyed first): never touch it here
    if (h->stream && h->stream == h->own_stream) cudaStreamSynchronize(h->own_stream); else cudaDeviceSynchronize();
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    for (auto e : h->ev) cudaEventDestroy(e);
    if (h->arena) cudaFree(h->arena);
    if (h->h_err) cudaFreeHost(h->h_err);
    delete h;
}

int sslpl_orb_tables(const sslpl_orb* h, float* scale, float* invscale, float* sigma2, float* invsigma2, int* nfeat, int* umax16) {
    SSLPL_REQUIRE(h, SSLPL_ERR_ARG, "null handle");
    for (int i = 0; i < h->p.nlevels; i++) {
        if (scale) scale[i] = h->scale[i];
        if (invscale) invscale[i] = h->invscale[i];
        if (sigma2) sigma2[i] = h->sigma2[i];
        if (invsigma2) invsigma2[i] = h->invsigma2[i];
        if (nfeat) nfeat[i] = h->nfeat[i];
    }
    if (umax16) for (int i = 0; i < 16; i++) umax16[i] = h->umax[i];
    return SSLPL_OK;
}

int sslpl_orb_tables_host(int nfeatures, float scaleFactor, int nlevels, float* scale, float* invscale, float* sigma2, float* invsigma2, int* nfeat, int* umax16) {
    SSLPL_REQUIRE(nlevels >= 1 && nlevels <= SSLPL_MAX_LEVELS && nfeatures >= 1 && scaleFactor > 1.0f, SSLPL_ERR_ARG, "bad extractor parameters");
    sslpl_orb tmp;
    tmp.p.nfeatures = nfeatures; tmp.p.scaleFactor = scaleFactor; tmp.p.nlevels = nlevels;
    make_tables(&tmp);
    return sslpl_orb_tables(&tmp, scale, invscale, sigma2, invsigma2, nfeat, umax16);
}

int sslpl_orb_max_keypoints(const sslpl_orb* h) {
    if (!h) return 0;
    int s = 0; for (int l = 0; l < h->p.nlevels; l++) s += h->nfeat[l] + 16;
    return s;
}

int sslpl_orb_extract_batch_device(sslpl_orb* h, const uint8_t* d_imgs, int nframes, int width, int height, int pitch, size_t frame_stride) {
    SSLPL_REQUIRE(h && d_imgs, SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(nframes >= 1 && nframes <= h->p.max_batch, SSLPL_ERR_ARG, "nframes exceeds the handle's max_batch");
    SSLPL_REQUIRE(pitch >= width, SSLPL_ERR_ARG, "pitch < width");
    SSLPL_CUDA(cudaSetDevice(h->p.device));
    int rc = configure(h, width, height);
    if (rc) return rc;
    h->view.base = d_imgs; h->view.pitch = pitch; h->view.frame_stride = (long long)frame_stride;
    h->cur_frames = nframes;
    return run_pipeline(h, nframes);
}

int sslpl_orb_device_results(sslpl_orb* h, const sslpl_keypoint** d_kps, const uint8_t** d_desc, const int** d_n, int* cap) {
    SSLPL_REQUIRE(h, SSLPL_ERR_ARG, "null handle");
    if (d_kps) *d_kps = h->ws.kps;
    if (d_desc) *d_desc = h->ws.desc;
    if (d_n) *d_n = h->ws.nkp;
    if (cap) *cap = h->g.kp_total_cap ? h->g.kp_total_cap : sslpl_orb_max_keypoints(h);
    return SSLPL_OK;
}

int sslpl_orb_sync(sslpl_orb* h) {
    SSLPL_REQUIRE(h, SSLPL_ERR_ARG, "null handle");
    SSLPL_CUDA(cudaSetDevice(h->p.device));
    return check_device_err(h);
}

void* sslpl_orb_stream(sslpl_orb* h) { return h ? (void*)h->stream : nullptr; }

int sslpl_orb_set_stream(sslpl_orb* h, void* cuda_stream) {
    SSLPL_REQUIRE(h, SSLPL_ERR_ARG, "null handle");
    SSLPL_CUDA(cudaSetDevice(h->p.device));
    SSLPL_CUDA(cudaStreamSynchronize(h->stream));
    h->stream = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
    return SSLPL_OK;
}

// Enqueue H2D of the frames, the whole extraction and the D2H of the results on the handle's stream; no host sync.
static int orb_enqueue_host_batch(sslpl_orb* h, const uint8_t* imgs, int nframes, int width, int height, int pitch, size_t frame_stride,
                                  sslpl_keypoint* kps, uint8_t* desc, int cap, int* n, bool copy_results) {
    SSLPL_REQUIRE(nframes >= 1 && nframes <= h->p.max_batch, SSLPL_ERR_ARG, "nframes exceeds the handle's max_batch");
    SSLPL_REQUIRE(pitch >= width, SSLPL_ERR_ARG, "pitch < width");
    SSLPL_CUDA(cudaSetDevice(h->p.device));
    int rc = configure(h, width, height);
    if (rc) return rc;
    const int ip = (int)align_up(width, 16);
    const size_t fs = (size_t)ip * height;
    if (frame_stride == (size_t)pitch * height)
        SSLPL_CUDA(cudaMemcpy2DAsync(h->d_input, ip, imgs, pitch, width, (size_t)height * nframes, cudaMemcpyHostToDevice, h->stream));
    else
        for (int f = 0; f < nframes; f++)
            SSLPL_CUDA(cudaMemcpy2DAsync(h->d_input + f * fs, ip, imgs + f * frame_stride, pitch, width, height, cudaMemcpyHostToDevice, h->stream));
    h->view.base = h->d_input; h->view.pitch = ip; h->view.frame_stride = (long long)fs;
    h->cur_frames = nframes;
    rc = run_pipeline(h, nframes);
    if (rc) return rc;
    const int kc = h->g.kp_total_cap;
    SSLPL_CUDA(cudaMemcpyAsync(n, h->ws.nkp, sizeof(int) * nframes, cudaMemcpyDeviceToHost, h->stream));
    if (copy_results) {
        SSLPL_CUDA(cudaMemcpy2DAsync(kps, (size_t)cap * sizeof(sslpl_keypoint), h->ws.kps, (size_t)kc * sizeof(sslpl_keypoint),
                                     (size_t)kc * sizeof(sslpl_keypoint), nframes, cudaMemcpyDeviceToHost, h->stream));
        SSLPL_CUDA(cudaMemcpy2DAsync(desc, (size_t)cap * 32, h->ws.desc, (size_t)kc * 32, (size_t)kc * 32, nframes, cudaMemcpyDeviceToHost, h->stream));
    }
    return SSLPL_OK;
}

int sslpl_orb_extract_batch_begin(sslpl_orb* h, const uint8_t* imgs, int nframes, int width, int height, int pitch, size_t frame_stride,
                                  sslpl_keypoint* kps, uint8_t* desc, int cap, int* n) {
    SSLPL_REQUIRE(h && kps && desc && n && imgs && width > 0 && height > 0, SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(cap >= sslpl_orb_max_keypoints(h), SSLPL_ERR_CAPACITY, "the asynchronous form needs cap >= sslpl_orb_max_keypoints()");
    return orb_enqueue_host_batch(h, imgs, nframes, width, height, pitch, frame_stride, kps, desc, cap, n, true);
}

int sslpl_orb_extract_batch(sslpl_orb* h, const uint8_t* imgs, int nframes, int width, int height, int pitch, size_t frame_stride,
                            sslpl_keypoint* kps, uint8_t* desc, int cap, int* n) {
    SSLPL_REQUIRE(h && kps && desc && n, SSLPL_ERR_ARG, "null argument");
    if (!imgs || width <= 0 || height <= 0) { for (int f = 0; f < nframes; f++) n[f] = 0; return SSLPL_OK; }   // ORBextractor.cc:1046
    const bool fits = cap >= sslpl_orb_max_keypoints(h);
    int rc = orb_enqueue_host_batch(h, imgs, nframes, width, height, pitch, frame_stride, kps, desc, cap, n, fits);
    if (rc) return rc;
    rc = check_device_err(h);
    if (rc || fits) return rc;
    // caller capacity smaller than the worst case: counts are on the host now, download only what fits
    const int kc = h->g.kp_total_cap;
    for (int f = 0; f < nframes; f++) SSLPL_REQUIRE(n[f] <= cap, SSLPL_ERR_CAPACITY, "caller keypoint capacity too small");
    SSLPL_CUDA(cudaMemcpy2DAsync(kps, (size_t)cap * sizeof(sslpl_keypoint), h->ws.kps, (size_t)kc * sizeof(sslpl_keypoint),
                                 (size_t)cap * sizeof(sslpl_keypoint), nframes, cudaMemcpyDeviceToHost, h->stream));
    SSLPL_CUDA(cudaMemcpy2DAsync(desc, (size_t)cap * 32, h->ws.desc, (size_t)kc * 32, (size_t)cap * 32, nframes, cudaMemcpyDeviceToHost, h->stream));
    SSLPL_CUDA(cudaStreamSynchronize(h->stream));
    return SSLPL_OK;
}

int sslpl_orb_extract(sslpl_orb* h, const uint8_t* img, int width, int height, int pitch, sslpl_keypoint* kps, uint8_t* desc, int cap, int* n) {
    return sslpl_orb_extract_batch(h, img, 1, width, height, pitch, (size_t)pitch * height, kps, desc, cap, n);
}

int sslpl_orb_level_size(const sslpl_orb* h, int level, int* w, int* hgt) {
    SSLPL_REQUIRE(h && level >= 0 && level < h->p.nlevels && h->cur_w > 0, SSLPL_ERR_ARG, "bad level or no frame processed yet");
    *w = h->g.lv[level].w; *hgt = h->g.lv[level].h;
    return SSLPL_OK;
}

static int download_plane(sslpl_orb* h, const uint8_t* src, int spitch, int w, int hh, std::vector<uint8_t>& out) {
    out.resize((size_t)w * hh);
    SSLPL_CUDA(cudaMemcpy2DAsync(out.data(), w, src, spitch, w, hh, cudaMemcpyDeviceToHost, h->stream));
    SSLPL_CUDA(cudaStreamSynchronize(h->stream));
    return SSLPL_OK;
}

int sslpl_orb_download_level(sslpl_orb* h, int frame, int level, int bordered, uint8_t* dst, int dpitch) {
    SSLPL_REQUIRE(h && dst && level >= 0 && level < h->p.nlevels && frame >= 0 && frame < h->cur_frames, SSLPL_ERR_ARG, "bad argument");
    SSLPL_CUDA(cudaSetDevice(h->p.device));
    const LevelGeom& L = h->g.lv[level];
    const uint8_t* src = level == 0 ? h->view.base + (long long)frame * h->view.frame_stride
                                    : h->ws.pyr + (long long)frame * h->g.pyr_stride + L.img_off;
    const int sp = level == 0 ? h->view.pitch : L.pitch;
    std::vector<uint8_t> tmp;
    int rc = download_plane(h, src, sp, L.w, L.h, tmp);
    if (rc) return rc;
    const int b = bordered ? EDGE : 0;      // copyMakeBorder(BORDER_REFLECT_101), ORBextractor.cc:1122-1129 (host-side view only)
    auto refl = [](int p, int len) { if (len == 1) return 0; while (p < 0 || p >= len) p = p < 0 ? -p : 2 * len - 2 - p; return p; };
    for (int y = -b; y < L.h + b; y++)
        for (int x = -b; x < L.w + b; x++)
            dst[(size_t)(y + b) * dpitch + x + b] = tmp[(size_t)refl(y, L.h) * L.w + refl(x, L.w)];
    return SSLPL_OK;
}

int sslpl_orb_download_blurred(sslpl_orb* h, int frame, int level, uint8_t* dst, int dpitch) {
    SSLPL_REQUIRE(h && dst && level >= 0 && level < h->p.nlevels && frame >= 0 && frame < h->cur_frames, SSLPL_ERR_ARG, "bad argument");
    SSLPL_CUDA(cudaSetDevice(h->p.device));
    const LevelGeom& L = h->g.lv[level];
    SSLPL_CUDA(cudaMemcpy2DAsync(dst, dpitch, h->ws.blur + (long long)frame * h->g.blur_stride + L.blur_off, L.bpitch, L.w, L.h,
                                 cudaMemcpyDeviceToHost, h->stream));
    SSLPL_CUDA(cudaStreamSynchronize(h->stream));
    return SSLPL_OK;
}

int sslpl_orb_download_candidates(sslpl_orb* h, int frame, int level, int* xs, int* ys, int* resp, int cap, int* n) {
    SSLPL_REQUIRE(h && n && level >= 0 && level < h->p.nlevels && frame >= 0 && frame < h->cur_frames, SSLPL_ERR_ARG, "bad argument");
    SSLPL_CUDA(cudaSetDevice(h->p.device));
    const LevelGeom& L = h->g.lv[level];
    std::vector<int> cnt(std::max(L.ncells, 1));
    std::vector<uint32_t> cand((size_t)std::max(L.ncells, 1) * L.cell_cap);
    SSLPL_CUDA(cudaStreamSynchronize(h->stream));
    if (L.ncells) {
        SSLPL_CUDA(cudaMemcpy(cnt.data(), h->ws.cell_cnt + (long long)frame * h->g.total_cells + L.cell_base, sizeof(int) * L.ncells, cudaMemcpyDeviceToHost));
        SSLPL_CUDA(cudaMemcpy(cand.data(), h->ws.cand + (long long)frame * h->g.cand_stride + L.cand_off, sizeof(uint32_t) * cand.size(), cudaMemcpyDeviceToHost));
    }
    int k = 0;
    for (int c = 0; c < L.ncells; c++)
        for (int s = 0; s < cnt[c]; s++, k++)
            if (k < cap) { uint32_t v = cand[(size_t)c * L.cell_cap + s]; xs[k] = v & 0xfff; ys[k] = (v >> 12) & 0xfff; resp[k] = v >> 24; }
    *n = k;
    return SSLPL_OK;
}

int sslpl_orb_download_level_keypoints(sslpl_orb* h, int frame, int level, int* xs, int* ys, int* resp, int cap, int* n) {
    SSLPL_REQUIRE(h && n && level >= 0 && level < h->p.nlevels && frame >= 0 && frame < h->cur_frames, SSLPL_ERR_ARG, "bad argument");
    SSLPL_CUDA(cudaSetDevice(h->p.device));
    const LevelGeom& L = h->g.lv[level];
    int cnt = 0;
    SSLPL_CUDA(cudaStreamSynchronize(h->stream));
    SSLPL_CUDA(cudaMemcpy(&cnt, h->ws.lvl_cnt + frame * MAXL + level, sizeof(int), cudaMemcpyDeviceToHost));
    std::vector<uint32_t> kp(std::max(cnt, 1));
    if (cnt) SSLPL_CUDA(cudaMemcpy(kp.data(), h->ws.lvl_kp + (long long)frame * h->g.kp_total_cap + L.kp_base, sizeof(uint32_t) * cnt, cudaMemcpyDeviceToHost));
    for (int i = 0; i < cnt && i < cap; i++) { xs[i] = kp[i] & 0xfff; ys[i] = (kp[i] >> 12) & 0xfff; resp[i] = kp[i] >> 24; }
    *n = cnt;
    return SSLPL_OK;
}

long long sslpl_orb_launch_count(const sslpl_orb* h) { return h ? h->launches : 0; }

int sslpl_orb_set_profiling(sslpl_orb* h, int on) { SSLPL_REQUIRE(h, SSLPL_ERR_ARG, "null handle"); h->profiling = on != 0; return SSLPL_OK; }

int sslpl_orb_stage_ms(sslpl_orb* h, float* ms, int cap, const char** names, int* nstages) {
    SSLPL_REQUIRE(h && nstages, SSLPL_ERR_ARG, "null argument");
    SSLPL_CUDA(cudaStreamSynchronize(h->stream));
    int k = 0;
    for (int i = 1; i < h->ev_n; i++, k++)
        if (k < cap) { float t = 0; cudaEventElapsedTime(&t, h->ev[i - 1], h->ev[i]); if (ms) ms[k] = t; if (names) names[k] = h->ev_name[i]; }
    *nstages = k;
    return SSLPL_OK;
}

}  // extern "C"
