// line.cu — B200 (sm_100a) line path: LSD (OpenCV 4.13 LineSegmentDetector, LSD_REFINE_ADV) + KeyLine packaging +
// LBD 256-bit descriptors + line equations.  Replaces LineSegment::ExtractLineSegment
// (reference src/ExtractLineSegment.cpp:18-69, which delegates to cv::line_descriptor / cv::LineSegmentDetector).
//
// Per-pixel stages are ordinary data-parallel kernels (k_sep7, k_resize_exact, k_ll_angle, k_lsd_seeds, k_lsd_nfa_*, k_sobel).
// The region stage (k_lsd_regions) is order-dependent by definition (seeds in descending gradient bins, shared
// `used` map, incrementally updated region angle): one warp walks one frame; the warp's lanes cooperate on neighbour
// fetches and on the rectangle scans of rect_nfa, frames of a batch run on different SMs.  It is latency-bound,
// not HBM-bound, and is reported separately (SURVEY.md 7.3 item 1).
//
// This file is compiled with -fmad=false: every float/double expression is evaluated as separate IEEE operations,
// in the same order as the CPU restatement, so that discrete decisions (alignment tests, density, NFA) agree.
#include "common.cuh"
#include "mathx.cuh"
#include "ddtrig.h"
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdlib>
#include <vector>

namespace sslpl {

constexpr double L_PI = 3.14159265358979323846;
constexpr double L_DEG = L_PI / 180;
constexpr double L_3_2_PI = (3 * L_PI) / 2;
constexpr double L_2PI = 2 * L_PI;
constexpr float NOTDEF_F = -1024.f;
constexpr int NBINS = 1024;
constexpr int LT_W = 64, LT_H = 32;          // tile of the separable filter

struct LineGeom {
    int w, h, pitch;            // input frame (pitch of the staging / view)
    int bpitch;                 // blurred planes (7-tap for LSD, 5-tap for LBD)
    int sw, sh, spitch;         // LSD detection scale (0.8x)
    int tiles_x, tiles_y;
    int xtab_off, ytab_off;     // INTER_LINEAR_EXACT tables (int2: index, w1)
    int seg_cap;                // raw segments per frame
    int kl_cap;                 // lsdNFeatures
    long long in_stride, blur_stride, scaled_stride, pix_stride /* sw*sh */, full_stride /* w*h */;
    double rho, prec, p, log_nt;
    int min_reg_size;
    int trace_cap;              // rows of the debug trace per frame (0 = off)
    int dbg;                    // SSLPL_WALKER_DBG bit mask (bring-up switches of the region walker)
};

// What region growing reads per neighbour, in one 16-byte load: level-line angle (degrees, NOTDEF_F when undefined),
// (float)cos / sin of (float)(angle in radians) — the values region_grow sums — and the mutable `used` flag.
// `used`: 0 = free.  The multi-warp walker stores the ticket of the region-growing attempt holding the pixel, the one-warp walker 1.
struct __align__(16) LPix { float ang, cx, cy; unsigned used; };

struct LineWs {
    uint8_t* blur7; uint8_t* blur5; uint8_t* scaled;
    float* angdeg; LPix* pix; float2* cs0; double* modgrad;
    unsigned long long* maxgrad; unsigned* seeds; int* nseeds;
    unsigned* reg;              // region pixel list (x | y << 16) of the turn holder (whole-frame capacity)
    unsigned* sreg;             // per frame: WALK_RING speculation slots x WALK_SLOT_CAP list entries
    unsigned long long* wstat;  // walker statistics (whole launch): see sslpl_line_walker_stats
    double* seg;                // raw rectangles: x1,y1,x2,y2 (detection scale, before +0.5)
    int* nseg;
    double* jobs; int* njobs; int* jobflag;   // NFA jobs: 13 doubles per candidate region (LRect + log_nfa), in walker order
    int2* jobnk; double* jobnfa;              // per job: (total, aligned) pixel counts and NFA of the unmodified rectangle
    int2* rej; int* rejctl;                   // work list of rejected jobs (frame, job); rejctl[0] = count, rejctl[1] = cursor, rejctl[2] = walker frame cursor
    int16_t* dx; int16_t* dy;
    int2* tab;
    float* resp; float4* ext;   // per raw segment: response and clamped extremes
    sslpl_keyline* kl; uint8_t* ldesc; double* lineeq; int* nl;
    int* err;
    double* trace; int* ntrace;
    const double* lgam;         // lgam[n] = log_gamma(n + 1) of lsd.cpp (Lanczos / Windschitl), tabulated by the host's libm
};

struct LView { const uint8_t* base; int pitch; long long frame_stride; };

// -------------------------------------------------------------------------------------------------
// Separable fixed-point filter (OpenCV 4.13 GaussianBlur 8U path): out = (sum_j k_j sum_i k_i p + 32768) >> 16
// taps are passed as 7 ints (5-tap kernels are zero-padded), BORDER_REFLECT_101.
// -------------------------------------------------------------------------------------------------
struct Taps7 { int k[7]; };

// Packed arithmetic: the horizontal pass is two dp4a per output on byte windows cut out of three aligned words with funnel
// shifts; its u16 results are stored as vertical PAIRS (row r | row r+1 << 16) so that the vertical pass is four dp2a per
// output.  All taps are < 256 and every partial sum < 65536, so the packed forms are exact.
// One launch filters the SAME staged input tile with two tap sets (LSD's 7-tap pre-blur and the 5-tap blur of the LBD stage): the tile
// is read from global memory once (round 2b; two launches of the one-filter form before).  out1 == nullptr: one filter only.
__global__ void __launch_bounds__(256) k_sep7(const __grid_constant__ LineGeom g, LView v, uint8_t* out0, uint8_t* out1, long long out_stride, Taps7 t0, Taps7 t1) {
    constexpr int IW = LT_W + 6, IP = LT_W + 8, IH = LT_H + 6;           // IP % 4 == 0: rows of s_in are word aligned
    __shared__ __align__(4) uint8_t s_in[IH * IP];
    __shared__ __align__(16) unsigned s_pair[IH * LT_W];                 // [r][x] = row r | row r+1 << 16
    unsigned short* s_half = reinterpret_cast<unsigned short*>(s_pair);
    const int tile = blockIdx.x, f = blockIdx.y, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int ty = tile / g.tiles_x, tx = tile - ty * g.tiles_x, x0 = tx * LT_W, y0 = ty * LT_H;
    const uint8_t* img = v.base + f * v.frame_stride;
    for (int yy = wid; yy < IH; yy += 8) {                               // a warp per input row: no per-element division
        const uint8_t* src = img + (long long)reflect101(y0 + yy - 3, g.h) * v.pitch;
        for (int xx = lane; xx < IW; xx += 32) s_in[yy * IP + xx] = __ldg(src + reflect101(x0 + xx - 3, g.w));
    }
    __syncthreads();
#pragma unroll 1
    for (int pass = 0; pass < 2; pass++) {
        uint8_t* out = pass ? out1 : out0;
        if (!out) break;
        const Taps7& t = pass ? t1 : t0;
        const unsigned T0 = (unsigned)t.k[0] | ((unsigned)t.k[1] << 8) | ((unsigned)t.k[2] << 16) | ((unsigned)t.k[3] << 24);
        const unsigned T1 = (unsigned)t.k[4] | ((unsigned)t.k[5] << 8) | ((unsigned)t.k[6] << 16);
        for (int i = tid; i < IH * (LT_W / 4); i += 256) {
            const int yy = i / (LT_W / 4), x4 = (i - yy * (LT_W / 4)) * 4;
            const unsigned* w = reinterpret_cast<const unsigned*>(&s_in[yy * IP + x4]);
            const unsigned w0 = w[0], w1 = w[1], w2 = w[2];                  // bytes x4 .. x4+11 (output k uses bytes k .. k+6)
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const unsigned A = k ? __funnelshift_r(w0, w1, 8 * k) : w0, B = k ? __funnelshift_r(w1, w2, 8 * k) : w1;
                const unsigned r = __dp4a(A, T0, __dp4a(B, T1, 0u));
                s_half[(yy * LT_W + x4 + k) * 2] = (unsigned short)r;                          // low half of pair row yy
                if (yy > 0) s_half[((yy - 1) * LT_W + x4 + k) * 2 + 1] = (unsigned short)r;    // high half of pair row yy-1
            }
        }
        __syncthreads();
        uint8_t* o = out + f * out_stride;
        const unsigned C01 = (unsigned)t.k[0] | ((unsigned)t.k[1] << 8), C23 = (unsigned)t.k[2] | ((unsigned)t.k[3] << 8);
        const unsigned C45 = (unsigned)t.k[4] | ((unsigned)t.k[5] << 8), C6 = (unsigned)t.k[6];
        for (int i = tid; i < LT_H * (LT_W / 4); i += 256) {
            const int yy = i / (LT_W / 4), x4 = (i - yy * (LT_W / 4)) * 4;
            if (y0 + yy >= g.h || x0 + x4 >= g.w) continue;
            const uint4 p0 = *reinterpret_cast<const uint4*>(&s_pair[yy * LT_W + x4]), p2 = *reinterpret_cast<const uint4*>(&s_pair[(yy + 2) * LT_W + x4]);
            const uint4 p4 = *reinterpret_cast<const uint4*>(&s_pair[(yy + 4) * LT_W + x4]), p6 = *reinterpret_cast<const uint4*>(&s_pair[(yy + 6) * LT_W + x4]);
            const unsigned a0 = __dp2a_lo(p0.x, C01, __dp2a_lo(p2.x, C23, __dp2a_lo(p4.x, C45, __dp2a_lo(p6.x, C6, 32768u))));
            const unsigned a1 = __dp2a_lo(p0.y, C01, __dp2a_lo(p2.y, C23, __dp2a_lo(p4.y, C45, __dp2a_lo(p6.y, C6, 32768u))));
            const unsigned a2 = __dp2a_lo(p0.z, C01, __dp2a_lo(p2.z, C23, __dp2a_lo(p4.z, C45, __dp2a_lo(p6.z, C6, 32768u))));
            const unsigned a3 = __dp2a_lo(p0.w, C01, __dp2a_lo(p2.w, C23, __dp2a_lo(p4.w, C45, __dp2a_lo(p6.w, C6, 32768u))));
            *reinterpret_cast<uint32_t*>(o + (long long)(y0 + yy) * g.bpitch + x0 + x4) = (a0 >> 16) | ((a1 >> 16) << 8) | ((a2 >> 16) << 16) | ((a3 >> 16) << 24);
        }
        __syncthreads();                                                  // s_pair is rewritten by the second filter
    }
}

// cv::resize(INTER_LINEAR_EXACT) 8U, 8.8 fixed point (SURVEY.md A.6 iii): tables hold (i0, w1)
__global__ void __launch_bounds__(256) k_resize_exact(const __grid_constant__ LineGeom g, LineWs ws) {
    const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y, f = blockIdx.z;
    if (x >= g.sw || y >= g.sh) return;
    const uint8_t* S = ws.blur7 + f * g.blur_stride;
    const int2 tx = __ldg(&ws.tab[g.xtab_off + x]), ty = __ldg(&ws.tab[g.ytab_off + y]);
    const int i0 = tx.x, i1 = min(i0 + 1, g.w - 1), w1 = tx.y, w0 = 256 - w1;
    const uint8_t* S0 = S + (long long)ty.x * g.bpitch;
    const uint8_t* S1 = S + (long long)min(ty.x + 1, g.h - 1) * g.bpitch;
    const int r0 = w0 * __ldg(S0 + i0) + w1 * __ldg(S0 + i1), r1 = w0 * __ldg(S1 + i0) + w1 * __ldg(S1 + i1);
    const int v1 = ty.y, v0 = 256 - v1;
    ws.scaled[f * g.scaled_stride + (long long)y * g.spitch + x] = (uint8_t)((v0 * r0 + v1 * r1 + 32768) >> 16);
}

// sin / cos of x in [0, 2 pi] to ~1 ulp (double): Cody-Waite reduction by pi/2 and the fdlibm kernel polynomials.
// Branch-free and table-free (libm's sincos drags its large-argument path and constant-bank tables through the
// memory pipe); the callers round the results to float, which hides the last-ulp freedom.
__device__ __forceinline__ void l_sincos_2pi(double x, double* s_out, double* c_out) {
    const double k = rint(x * 0.6366197723675814);
    const double r = (x - k * 1.57079632673412561417e+00) - k * 6.07710050650619224932e-11;
    const double z = r * r;
    double ps = 1.58969099521155010221e-10;
    ps = -2.50507602534068634195e-08 + z * ps; ps = 2.75573137070700676789e-06 + z * ps; ps = -1.98412698298579493134e-04 + z * ps;
    ps = 8.33333333332248946124e-03 + z * ps; ps = -1.66666666666666324348e-01 + z * ps;
    const double s = r + r * (z * ps);
    double pc = -1.13596475577881948265e-11;
    pc = 2.08757232129817482790e-09 + z * pc; pc = -2.75573143513906633035e-07 + z * pc; pc = 2.48015872894767294178e-05 + z * pc;
    pc = -1.38888888888741095749e-03 + z * pc; pc = 4.16666666666666019037e-02 + z * pc;
    const double c = (1.0 - 0.5 * z) + z * (z * pc);
    const int q = (int)k & 3;
    *s_out = (q == 0) ? s : (q == 1) ? c : (q == 2) ? -s : -c;
    *c_out = (q == 0) ? c : (q == 1) ? -s : (q == 2) ? -c : s;
}

// ll_angle (lsd.cpp): 2x2 gradient, level-line angle, gradient norm, max over defined pixels
// Four horizontally adjacent pixels per thread: 4 loads and 9 vector stores per 4 pixels instead of 16 + 16 (the
// scalar version was limited by the memory-instruction queue, not by HBM or by the trigonometry).
__global__ void __launch_bounds__(256) k_ll_angle(const __grid_constant__ LineGeom g, LineWs ws) {
    const int x0 = (blockIdx.x * 32 + threadIdx.x) * 4, y = blockIdx.y * 8 + threadIdx.y, f = blockIdx.z;
    unsigned long long bits = 0ull;                    // max gradient norm of the defined pixels (positive doubles order like integers)
    if (x0 < g.sw && y < g.sh) {
        float ang[4]; float2 cs[4], cs0[4]; double norm[4];
        const uint8_t* p = ws.scaled + f * g.scaled_stride + (long long)y * g.spitch + x0;
        unsigned r0 = 0, r1 = 0; int e0 = 0, e1 = 0;    // rows y, y+1: bytes x0..x0+3 and x0+4
        const bool row_ok = y < g.sh - 1;
        if (row_ok) {
            r0 = *reinterpret_cast<const unsigned*>(p); r1 = *reinterpret_cast<const unsigned*>(p + g.spitch);   // spitch % 64 == 0, x0 % 4 == 0
            if (x0 + 4 < g.sw) { e0 = p[4]; e1 = p[g.spitch + 4]; }
        }
#pragma unroll
        for (int k = 0; k < 4; k++) {
            ang[k] = NOTDEF_F; cs[k] = make_float2(0.f, 0.f); cs0[k] = make_float2(0.f, 0.f); norm[k] = 0;
            if (row_ok && x0 + k < g.sw - 1) {
                const int A = (r0 >> (8 * k)) & 0xff, C = (r1 >> (8 * k)) & 0xff;
                const int Bv = (k < 3) ? (int)((r0 >> (8 * k + 8)) & 0xff) : e0, D = (k < 3) ? (int)((r1 >> (8 * k + 8)) & 0xff) : e1;
                const int DA = D - A, BC = Bv - C;
                const int gx = DA + BC, gy = DA - BC;
                norm[k] = sqrt((double)(gx * gx + gy * gy) / 4.0);
                if (norm[k] > g.rho) {
                    const unsigned long long nb = (unsigned long long)__double_as_longlong(norm[k]);
                    bits = nb > bits ? nb : bits;
                    ang[k] = fast_atan2_deg((float)gx, (float)-gy);
                    const double ad = (double)ang[k] * L_DEG;
                    const float a = (float)ad;
                    double sn, cn;
                    l_sincos_2pi((double)a, &sn, &cn);
                    cs[k].x = (float)cn; cs[k].y = (float)sn;
                    // region_grow's seed values float(cos(ad)), float(sin(ad)): ad = a + d with |d| < 2e-7, so a second-order
                    // Taylor step from (cn, sn) is accurate to a few double ulps (the d^3 term is < 1e-20) — one sincos, not four calls
                    const double d = ad - (double)a, hd2 = 0.5 * d * d;
                    cs0[k].x = (float)(cn - sn * d - cn * hd2); cs0[k].y = (float)(sn + cn * d - sn * hd2);
                }
            }
        }
        const long long pi = f * g.pix_stride + (long long)y * g.sw + x0;
        if ((g.sw & 3) == 0 && (g.pix_stride & 3) == 0) {                  // rows start 16-byte aligned in every per-pixel array
            *reinterpret_cast<float4*>(ws.angdeg + pi) = make_float4(ang[0], ang[1], ang[2], ang[3]);
            float4* c4 = reinterpret_cast<float4*>(ws.cs0 + pi);
            c4[0] = make_float4(cs0[0].x, cs0[0].y, cs0[1].x, cs0[1].y); c4[1] = make_float4(cs0[2].x, cs0[2].y, cs0[3].x, cs0[3].y);
            double2* m2 = reinterpret_cast<double2*>(ws.modgrad + pi);
            m2[0] = make_double2(norm[0], norm[1]); m2[1] = make_double2(norm[2], norm[3]);
            uint4* px = reinterpret_cast<uint4*>(ws.pix + pi);
#pragma unroll
            for (int k = 0; k < 4; k++) px[k] = make_uint4(__float_as_uint(ang[k]), __float_as_uint(cs[k].x), __float_as_uint(cs[k].y), 0u);
        } else {
#pragma unroll
            for (int k = 0; k < 4; k++) if (x0 + k < g.sw) {
                ws.angdeg[pi + k] = ang[k]; ws.cs0[pi + k] = cs0[k]; ws.modgrad[pi + k] = norm[k];
                LPix px; px.ang = ang[k]; px.cx = cs[k].x; px.cy = cs[k].y; px.used = 0u;
                ws.pix[pi + k] = px;
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { const unsigned long long t = __shfl_xor_sync(0xffffffffu, bits, o); bits = t > bits ? t : bits; }
    if ((threadIdx.x & 31) == 0 && bits) atomicMax(ws.maxgrad + f, bits);
}

__device__ __forceinline__ int lsd_bin(double norm, double max_grad) {
    const double bin_coef = (max_grad > 0) ? double(NBINS - 1) / max_grad : 0;
    return (int)(norm * bin_coef);
}

// Seed ordering of lsd.cpp in one kernel: the defined pixels sorted by gradient bin (descending), raster order inside
// a bin — a stable counting sort.  One CTA of 32 warps per frame; warp w owns the w-th contiguous pixel range (raster
// order), builds its own 1024-bin histogram in shared memory, the histograms are prefix-summed across warps and bins,
// and every warp then scatters its pixels in order (ranks inside a 32-group by __match_any_sync).
constexpr int SEED_WARPS = 8;                       // warps per frame: 32 KB of histograms and ~16k registers per CTA, so that
                                                    // seed CTAs fit on SMs that are busy with region walkers of other batches
__global__ void __launch_bounds__(SEED_WARPS * 32) k_lsd_seeds(const __grid_constant__ LineGeom g, LineWs ws) {
    __shared__ int s_wh[SEED_WARPS * NBINS];         // [warp][bin] running offsets
    __shared__ int s_warp[33];
    constexpr int NT = SEED_WARPS * 32, BPT = NBINS / NT;   // bins per thread in the prefix step
    const int f = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    // a pixel is defined (angle != NOTDEF) exactly when its gradient norm exceeds rho (k_ll_angle): one array to read
    const double* mod = ws.modgrad + f * g.pix_stride;
    const double mg = __longlong_as_double((long long)ws.maxgrad[f]), rho = g.rho;
    const double bin_coef = (mg > 0) ? double(NBINS - 1) / mg : 0;
    int* wh = s_wh + wid * NBINS;
    for (int i = tid; i < SEED_WARPS * NBINS; i += NT) s_wh[i] = 0;
    __syncthreads();
    const long long per = ((g.pix_stride + SEED_WARPS - 1) / SEED_WARPS + 31) / 32 * 32;   // pixels per warp, multiple of 32
    const long long b = wid * per, e = min(g.pix_stride, b + per);
    constexpr int U = 8;                                                       // groups of 32 pixels in flight per warp
    for (long long i0 = b; i0 < e; i0 += 32 * U) {
        double m[U];
#pragma unroll
        for (int u = 0; u < U; u++) { const long long i = i0 + u * 32 + lane; m[u] = i < e ? __ldg(mod + i) : 0.0; }
#pragma unroll
        for (int u = 0; u < U; u++) if (m[u] > rho) atomicAdd(&wh[NBINS - 1 - (int)(m[u] * bin_coef)], 1);
    }
    __syncthreads();
    {   // thread = BPT consecutive bins: exclusive prefix over the warps inside each bin, then over the bins
        int run[BPT], mine = 0;
#pragma unroll
        for (int k = 0; k < BPT; k++) {
            const int bin = tid * BPT + k;
            int r = 0;
            for (int w = 0; w < SEED_WARPS; w++) { const int c = s_wh[w * NBINS + bin]; s_wh[w * NBINS + bin] = r; r += c; }
            run[k] = r; mine += r;
        }
        int total;
        int base = block_exclusive_scan(mine, s_warp, &total);
#pragma unroll
        for (int k = 0; k < BPT; k++) {
            const int bin = tid * BPT + k;
            for (int w = 0; w < SEED_WARPS; w++) s_wh[w * NBINS + bin] += base;
            base += run[k];
        }
        if (tid == 0) ws.nseeds[f] = total;
    }
    __syncthreads();
    unsigned* seeds = ws.seeds + f * g.pix_stride;
    for (long long i0 = b; i0 < e; i0 += 32 * U) {
        double m[U];
#pragma unroll
        for (int u = 0; u < U; u++) { const long long i = i0 + u * 32 + lane; m[u] = i < e ? __ldg(mod + i) : 0.0; }
#pragma unroll
        for (int u = 0; u < U; u++) {                                          // groups in raster order: a stable sort
            const bool def = m[u] > rho;
            if (!__any_sync(0xffffffffu, def)) continue;
            const int key = def ? (NBINS - 1 - (int)(m[u] * bin_coef)) : (2048 + lane);
            const unsigned peers = __match_any_sync(0xffffffffu, key);
            const int leader = __ffs(peers) - 1, rank = __popc(peers & ((1u << lane) - 1));
            int off = 0;
            if (def && lane == leader) { off = wh[key]; wh[key] = off + __popc(peers); }
            off = __shfl_sync(0xffffffffu, off, leader);
            if (def) seeds[off + rank] = (unsigned)(i0 + u * 32 + lane);
            __syncwarp();
        }
    }
}

// -------------------------------------------------------------------------------------------------
// The sequential region walker.  All lanes run the same control flow on warp-uniform values; loads of 32
// region points / 9 neighbours are spread over the lanes and broadcast with shuffles; lane 0 does the writes.
// The walker's CTA is ONE warp; its per-frame context lives in shared memory (file scope) so that the big
// per-region routines can be real calls (__noinline__): inlined, the kernel was ~175 KB of SASS and the resident
// warps (each at a different place in it) spent most of their stall time on instruction fetch.
// -------------------------------------------------------------------------------------------------
struct LRect { double x1, y1, x2, y2, width, x, y, theta, dx, dy, prec, p; };

struct Walk {                   // context of the rectangle scans (k_lsd_nfa_*): registers
    int w, h;
    const float* ang;
    double log_nt;
    const double* lgam;
    int lane;
};

constexpr int WALK_MAXW = 16;          // warps of a walker CTA (one CTA per frame)
constexpr int WALK_RING = 64;          // region-growing attempts in flight per frame (speculation slots)
constexpr int WALK_SLOT_CAP = 2048;    // list entries of a slot: every pixel the attempt ever accepted + the pixels it assumed used
constexpr int WALK_SMALL = 32;         // attempts with at most this many list entries are committed from shared memory
constexpr int WALK_WIN = 64;           // seeds staged in shared memory for the claims

struct WalkCtx {                // context of one walker warp (k_lsd_regions): shared memory
    int w, h;
    const float* ang; const double* mod;
    LPix* pix;                  // packed per-pixel record; .used holds the ticket (global): who is growing over this pixel right now
    const unsigned* bits;       // the frame's COMMITTED `used` bitmap (shared memory); bits only ever go 0 -> 1
    unsigned* reg;              // current region list (x | y << 16)
    unsigned* base0;            // start of this attempt's list space
    const float2* cs0;          // per pixel: (float)cos / sin of the level-line angle taken as double (region seed values)
    int cap;                    // entries available at reg (the assumed-used list grows down from reg + cap)
    int nasm;                   // assumed-used pixels recorded so far
    int acc;                    // entries of base0[] that hold accepted-ever pixels (validated at commit)
    int seq;                    // rank of this attempt (claim order)
    int mode;                   // 0 = speculative, 1 = turn holder (everything of lower rank is committed)
    int dbg;
    int abort;                  // speculative attempt abandoned: 1 = capacity, 2 = a live attempt of LOWER rank holds a pixel it needs
    int conflict;               // abort == 2: that rank (the attempt can be repeated once it has been retired)
    unsigned ticket;
};
struct FrameCtl {               // one per walker CTA
    unsigned cursor, nclaims, turn;
    int claim_lock, commit_lock, all_claimed, nj, frame, ns, win_base;
    unsigned win[WALK_WIN];
    int seqof[WALK_RING], seedpix[WALK_RING], state[WALK_RING], acc[WALK_RING], nasm[WALK_RING], finoff[WALK_RING], nfin[WALK_RING], job[WALK_RING], poison[WALK_RING];
    double jobv[WALK_RING][13];                 // the pending NFA job of the slot
    unsigned small[WALK_RING][WALK_SMALL];      // acc + nasm <= WALK_SMALL and finoff == 0: accepted list, then the assumed pixels (as indices)
};
__shared__ WalkCtx s_Wc[WALK_MAXW];
__shared__ FrameCtl s_F;
__shared__ __align__(16) double s_stc[WALK_MAXW][96];     // per warp: staging of a 32-point chunk: 3 quantities x 32
__shared__ WalkCtx s_W1;                                   // the one-warp throughput kernel keeps its own small context:
__shared__ __align__(16) double s_st1[96];                 // 28 of its CTAs share an SM
constexpr int SOLO = 0;                                    // (hidden by the template parameter of the same name inside the helpers)
// SOLO: 0 = multi-warp walker (k_lsd_regions), 1 = one warp per frame (k_lsd_regions_solo)
#define s_W (*(SOLO == 1 ? &s_W1 : &s_Wc[threadIdx.x >> 5]))
#define s_st (SOLO == 1 ? s_st1 : s_stc[threadIdx.x >> 5])

// SLOT_PRESUMED: the seed was under the ticket of a live attempt of lower rank when its turn to be grown came: it is presumed
// swallowed; the commit checks (and grows it for real if it was not).  SLOT_ABORTED: to be redone by the turn holder.
enum { SLOT_EMPTY = 0, SLOT_RUNNING = 1, SLOT_DONE = 2, SLOT_ABORTED = 3, SLOT_PRESUMED = 4 };

// ticket = rank + 1 in bits 0..23, attempt number in bits 24..30, bit 31 = grown by the turn holder
__device__ __forceinline__ unsigned l_turn() { return *reinterpret_cast<volatile unsigned*>(&s_F.turn); }
__device__ __forceinline__ bool l_bit(const unsigned* bits, int q) { return (reinterpret_cast<const volatile unsigned*>(bits)[q >> 5] >> (q & 31)) & 1u; }
// Is ticket m (not mine) held by an attempt that has not been retired yet?  Ranks below `turn` are committed or discarded.
__device__ __forceinline__ bool l_live(unsigned m, int* seq_out) { const int s = (int)(m & 0xffffffu) - 1; *seq_out = s; return m != 0u && s >= (int)l_turn(); }
template <int SOLO> __device__ __forceinline__ void l_release(const WalkCtx& W, int q) {
    if (SOLO == 1) W.pix[q].used = 0u;
    else atomicCAS(&W.pix[q].used, W.ticket, 0u);
}

__device__ __forceinline__ bool l_aligned(float angdeg, double theta, double prec) {
    if (angdeg == NOTDEF_F) return false;
    const double a = (double)angdeg * L_DEG;
    double n = theta - a;
    if (n < 0) n = -n;
    if (n > L_3_2_PI) { n -= L_2PI; if (n < 0) n = -n; }
    return n <= prec;
}

__device__ __forceinline__ bool l_aligned_rad(double a, double theta, double prec) {      // a = (double)angdeg * L_DEG, not NOTDEF
    double n = theta - a;
    if (n < 0) n = -n;
    if (n > L_3_2_PI) { n -= L_2PI; if (n < 0) n = -n; }
    return n <= prec;
}

// region_grow (lsd.cpp).  FOUR queue entries are expanded per step: lane = 8 * slot + neighbour (the centre pixel is
// always used, so the 3x3 scan has 8 live neighbours, kept in the reference's yy-outer / xx-inner order), i.e. the 32
// lanes hold the next 32 neighbour tests of the sequential algorithm in order.  Sequential semantics (each neighbour
// is tested once, in scan order, against the region angle as updated by the neighbours accepted before it) are kept
// in as many rounds as there are acceptances: all pending lanes test against the current angle; the first passing
// lane k0 is accepted, lanes < k0 are definitively rejected (they saw exactly the angle the sequential scan would have
// shown them), later lanes holding the same pixel drop out (the scan would find it used).
//
// "Used" is what the sequential algorithm would see: the frame's committed bitmap (regions of lower rank that are final) or
// my own ticket.  A pixel under the ticket of a LIVE attempt of lower rank is assumed used and recorded (checked at commit);
// one under a live ticket of higher rank counts as free (taking it poisons that attempt).  A pixel is taken with one atomic
// whose result is only looked at one step later (the round trip overlaps the next step's loads): a speculative attempt that
// lost a pixel to a live attempt of lower rank is abandoned then (abort = 2, conflict = that rank).
// Returns -1 when the attempt has to be abandoned (s_W.abort says why).
struct LTake { unsigned seen, old; int q; bool pend; };
__device__ __forceinline__ void l_take_issue(const WalkCtx& W, LTake& t, int q, unsigned seen) {
    t.q = q; t.seen = seen; t.pend = true;
    t.old = W.mode == 0 ? atomicCAS(&W.pix[q].used, seen, W.ticket) : atomicExch(&W.pix[q].used, W.ticket);
}
// Looks at the result of the atomic issued one step earlier.  Returns -1 when the pixel is mine, the rank of the live attempt of
// LOWER rank that holds it (the speculative attempt must be repeated after that rank retires), or -2 when a speculative attempt lost
// the compare-and-swap to anybody else: the word changed between this attempt's read and its atomic, so other lanes may have acted
// on the stale ticket during the step in between (the pixel could be in the list twice) — the attempt is simply repeated at once.
__device__ __forceinline__ int l_take_resolve(const WalkCtx& W, LTake& t) {
    if (!t.pend) return -1;
    t.pend = false;
    const unsigned old = t.old; int s;
    if (W.mode != 0 || old == t.seen) {                           // the pixel is mine; whoever held it alive (higher rank) is poisoned
        if (old != W.ticket && l_live(old, &s) && s != W.seq) s_F.poison[s % WALK_RING] = 1;
        return -1;
    }
    return (l_live(old, &s) && s < W.seq) ? s : -2;
}

template <int SOLO> __device__ __noinline__ int l_region_grow(int sx, int sy, double prec, double* reg_angle_out) {
    WalkCtx& W = s_W;
    const int lane = threadIdx.x & 31, w = W.w, h = W.h;
    LPix* pix = W.pix; unsigned* reg = W.reg; const unsigned* bits = W.bits;
    const unsigned T = W.ticket; const int myseq = W.seq; const bool spec = W.mode == 0;
    const int sq = sy * w + sx;                                   // 32-bit pixel indices (sw * sh < 2^31)
    LTake tk; tk.pend = false; tk.q = 0; tk.seen = 0u; tk.old = 0u;
    int failrank = -1;                                            // -1 fine, >= 0 rank to wait for, -2 repeat at once
    if (SOLO) { if (lane == 0) { reg[0] = (unsigned)sx | ((unsigned)sy << 16); pix[sq].used = 1u; } }
    else {
        int fail = 0;
        if (lane == 0) {
            reg[0] = (unsigned)sx | ((unsigned)sy << 16);
            const unsigned m0 = __ldcg(&pix[sq].used);
            int s0;
            if (m0 != T) {
                if (spec && l_live(m0, &s0) && s0 < myseq) fail = 3;          // an in-flight region of lower rank reached the seed first: presumed swallowed
                else { W.conflict = -1; l_take_issue(W, tk, sq, m0); const int r = l_take_resolve(W, tk); if (r >= 0) fail = 3; else if (r == -2) fail = 2; }
            }
        }
        fail = __shfl_sync(0xffffffffu, fail, 0);
        if (fail) { W.abort = fail; return -1; }
    }
    double reg_angle = (double)__ldg(W.ang + sq) * L_DEG;
    const float2 c0 = __ldg(W.cs0 + sq);
    float sumdx = c0.x, sumdy = c0.y;
    int n = 1, nasm = W.nasm;
    const int cap = W.cap;
    const int slot = lane >> 3, nb = (lane & 7) + ((lane & 7) >= 4 ? 1 : 0);   // neighbour 0..8 without the centre (4)
    const int ox = nb % 3 - 1, oy = nb / 3 - 1;
    __syncwarp();
    for (int i = 0; i < n;) {
        const int cnt = min(4, n - i);
        unsigned pk = 0, pkn = 0;
        if (slot < cnt) pk = reg[i + slot];
        const bool hasn = i + 4 + slot < n;                      // the next step's entries, where they already exist:
        if (hasn) pkn = reg[i + 4 + slot];                       // pull their neighbour records towards L2 now
        const int xx = (int)(pk & 0xffff) + ox, yy = (int)(pk >> 16) + oy, q = yy * w + xx;
        const bool valid = slot < cnt && (unsigned)xx < (unsigned)w && (unsigned)yy < (unsigned)h;
        {
            const int xn = (int)(pkn & 0xffff) + ox, yn = (int)(pkn >> 16) + oy;
            if (hasn && (unsigned)xn < (unsigned)w && (unsigned)yn < (unsigned)h)
                asm volatile("prefetch.global.L2 [%0];" :: "l"(pix + (yn * w + xn)));
        }
        uint4 v = make_uint4(__float_as_uint(NOTDEF_F), 0u, 0u, 0u);
        if (valid) v = SOLO ? *reinterpret_cast<const uint4*>(pix + q) : __ldcg(reinterpret_cast<const uint4*>(pix + q));   // record + ticket in one load (L2: the ticket is mutable)
        if (!SOLO) { const int r = l_take_resolve(W, tk); if (r != -1) failrank = (r >= 0 && r > failrank) ? r : (failrank >= 0 ? failrank : r); }   // last step's atomic, while this step's loads fly
        const float a = __uint_as_float(v.x), cx = __uint_as_float(v.y), cy = __uint_as_float(v.z);
        const unsigned m = v.w;
        bool cand = false, assumed = false;
        if (SOLO) cand = valid && a != NOTDEF_F && m == 0u;
        else if (valid && a != NOTDEF_F && m != T && !l_bit(bits, q)) {
            int s;
            if (spec && l_live(m, &s) && s < myseq) { assumed = true; if (W.dbg & 16) failrank = s > failrank ? s : failrank; }
            else cand = true;
        }
        const unsigned lt = (1u << lane) - 1u;
        const unsigned am = __ballot_sync(0xffffffffu, assumed);
        if (am) {                                                 // remember what was assumed: the commit checks these bits are set
            if (n + nasm + __popc(am) > cap) { W.abort = 1; return -1; }
            if (assumed) reg[cap - 1 - nasm - __popc(am & lt)] = (unsigned)q;
            nasm += __popc(am);
        }
        const double ad = (double)a * L_DEG;
        unsigned pending = __ballot_sync(0xffffffffu, cand);
        while (pending) {
            const bool mep = (pending >> lane) & 1u;
            const unsigned S0 = __ballot_sync(0xffffffffu, mep && l_aligned_rad(ad, reg_angle, prec));
            if (!S0) break;                                       // nobody passes at the current angle: all rejected
            if (n + nasm + __popc(S0) > cap) { W.abort = 1; return -1; }
            if ((S0 & (S0 - 1u)) == 0u) {
                // exactly one candidate: the plain sequential step
                const int k0 = __ffs(S0) - 1;
                const float kx = __shfl_sync(0xffffffffu, cx, k0), ky = __shfl_sync(0xffffffffu, cy, k0);
                const int q0 = __shfl_sync(0xffffffffu, q, k0);
                if (lane == k0) { reg[n] = (unsigned)xx | ((unsigned)yy << 16); if (SOLO) pix[q].used = 1u; else l_take_issue(W, tk, q, m); }
                n++;
                sumdx += kx; sumdy += ky;
                reg_angle = (double)fast_atan2_deg(sumdy, sumdx) * L_DEG;
                pending &= ~((2u << k0) - 1u);
                pending &= ~__ballot_sync(0xffffffffu, q == q0);  // the same pixel seen from another queue entry
                continue;
            }
            // Several candidates: SPECULATE that exactly the lanes passing at the current angle (first holder of each
            // pixel only) will be accepted.  Every lane then forms the running sums the sequential scan would hold when
            // it reaches that lane (ordered float adds over the earlier members), ONE SIMT atan2 gives every member's
            // "angle after me", each pending lane re-tests itself against the angle of the member just before it, and
            // the speculation is accepted up to the first lane whose verified outcome differs from the guess (that
            // lane's verified outcome is the true one, because everything before it was right).
            const unsigned peers = __match_any_sync(0xffffffffu, mep ? q : ~lane);
            const bool inS0 = (S0 >> lane) & 1u;
            const unsigned S = S0 & ~__ballot_sync(0xffffffffu, inS0 && (peers & S0 & lt) != 0u);
            const bool inS = (S >> lane) & 1u;
            float bx = sumdx, by = sumdy;
            for (unsigned Tm = S; Tm; Tm &= Tm - 1u) {
                const int mm = __ffs(Tm) - 1;
                const float mx = __shfl_sync(0xffffffffu, cx, mm), my = __shfl_sync(0xffffffffu, cy, mm);
                if (lane > mm) { bx += mx; by += my; }
            }
            const float ax = bx + cx, ay = by + cy;
            const double aft = (double)fast_atan2_deg(ay, ax) * L_DEG;
            const unsigned prevm = S & lt;
            double bef = __shfl_sync(0xffffffffu, aft, (31 - __clz(prevm)) & 31);
            if (!prevm) bef = reg_angle;
            const bool dup_e = (peers & S & lt) != 0u;            // an earlier member holds my pixel: the scan finds it used
            const bool actual = mep && !dup_e && l_aligned_rad(ad, bef, prec);
            const unsigned mism = __ballot_sync(0xffffffffu, mep && (actual != inS));
            int src; unsigned A;
            if (!mism) { A = S; src = 31 - __clz(S); }
            else {
                src = __ffs(mism) - 1;
                const unsigned acc = __ballot_sync(0xffffffffu, actual);
                A = (S & ((1u << src) - 1u)) | (acc & (1u << src));
            }
            if ((A >> lane) & 1u) { reg[n + __popc(A & lt)] = (unsigned)xx | ((unsigned)yy << 16); if (SOLO) pix[q].used = 1u; else l_take_issue(W, tk, q, m); }
            n += __popc(A);
            const float selx = actual ? ax : bx, sely = actual ? ay : by;
            const double sela = actual ? aft : bef;
            sumdx = __shfl_sync(0xffffffffu, selx, src); sumdy = __shfl_sync(0xffffffffu, sely, src);
            reg_angle = __shfl_sync(0xffffffffu, sela, src);
            if (!mism) break;                                     // every pending lane is resolved
            pending &= ~((2u << src) - 1u);
            pending &= ~__ballot_sync(0xffffffffu, mep && (peers & A) != 0u);   // later holders of accepted pixels
        }
        __syncwarp();
        if (!SOLO && spec && __any_sync(0xffffffffu, failrank != -1)) break;   // lost a pixel: stop growing now
        i += cnt;
    }
    if (SOLO) { *reg_angle_out = reg_angle; return n; }
    { const int r = l_take_resolve(W, tk); if (r != -1) failrank = (r >= 0 && r > failrank) ? r : (failrank >= 0 ? failrank : r); }
    const bool lostany = __any_sync(0xffffffffu, failrank != -1);
    failrank = __reduce_max_sync(0xffffffffu, failrank);          // the highest rank to wait for (-1 / -2 lanes do not count)
    W.nasm = nasm;
    if (lostany) { W.abort = 2; W.conflict = failrank >= 0 ? failrank : -1; return -1; }
    *reg_angle_out = reg_angle;
    return n;
}

__device__ __forceinline__ double l_angle_diff_signed(double a, double b) {
    double d = a - b;
    while (d <= -L_PI) d += L_2PI;
    while (d > L_PI) d -= L_2PI;
    return d;
}

// Sum of the three staged quantities of one chunk, in list order: lane c (c = lane % 3) owns accumulator c, so a
// point costs one shared load and one add per warp instead of three of each.
template <int SOLO> __device__ __noinline__ double l_chunk_sum(const double* sp, int m, double acc) {
    if (m == 32) {
        const double2* s2 = reinterpret_cast<const double2*>(sp);
#pragma unroll
        for (int j = 0; j < 16; j++) { const double2 v = s2[j]; acc += v.x; acc += v.y; }
    } else {
#pragma unroll 1
        for (int j = 0; j < m; j++) acc += sp[j];
    }
    return acc;
}

// region2rect + get_theta (lsd.cpp).  The weighted sums must be accumulated in list order to stay bit-identical with
// the CPU, but only the ADDS are sequential: each lane forms the products of its own point, stages them in shared
// memory, and lanes 0..2 (replicated over the warp) each walk one of the three staged rows.  The extents are exact
// min/max.
template <int SOLO> __device__ __noinline__ void l_region2rect(int n, double reg_angle, double prec, double p, LRect* out) {
    const int lane = threadIdx.x & 31, w = s_W.w;
    const unsigned* reg = s_W.reg; const double* __restrict__ mod = s_W.mod;
    double* s0 = s_st; double* s1 = s_st + 32; double* s2 = s_st + 64;
    const double* sp = s_st + (lane % 3) * 32;
    double acc = 0;
#pragma unroll 1
    for (int b = 0; b < n; b += 32) {
        const int i = b + lane;
        if (i < n) {
            const unsigned pk = reg[i]; const int rx = pk & 0xffff, ry = pk >> 16;
            const double wg = mod[ry * w + rx];
            s0[lane] = (double)rx * wg; s1[lane] = (double)ry * wg; s2[lane] = wg;
        }
        __syncwarp();
        acc = l_chunk_sum<SOLO>(sp, min(32, n - b), acc);
        __syncwarp();
    }
    double x = __shfl_sync(0xffffffffu, acc, 0), y = __shfl_sync(0xffffffffu, acc, 1);
    const double sum = __shfl_sync(0xffffffffu, acc, 2);
    x /= sum; y /= sum;
    acc = 0;
#pragma unroll 1
    for (int b = 0; b < n; b += 32) {
        const int i = b + lane;
        if (i < n) {
            const unsigned pk = reg[i]; const int rx = pk & 0xffff, ry = pk >> 16;
            const double wg = mod[ry * w + rx];
            const double dx = (double)rx - x, dy = (double)ry - y;
            s0[lane] = dy * dy * wg; s1[lane] = dx * dx * wg; s2[lane] = -(dx * dy * wg);      // Ixy -= v  ==  Ixy += -v
        }
        __syncwarp();
        acc = l_chunk_sum<SOLO>(sp, min(32, n - b), acc);
        __syncwarp();
    }
    const double Ixx = __shfl_sync(0xffffffffu, acc, 0), Iyy = __shfl_sync(0xffffffffu, acc, 1), Ixy = __shfl_sync(0xffffffffu, acc, 2);
    const double lambda = 0.5 * (Ixx + Iyy - sqrt((Ixx - Iyy) * (Ixx - Iyy) + 4.0 * Ixy * Ixy));
    double theta = (fabs(Ixx) > fabs(Iyy)) ? (double)fast_atan2_deg((float)(lambda - Ixx), (float)Ixy)
                                           : (double)fast_atan2_deg((float)Ixy, (float)(lambda - Iyy));
    theta *= L_DEG;
    if (fabs(l_angle_diff_signed(theta, reg_angle)) > prec) theta += L_PI;
    // correctly-rounded cos/sin (see ddtrig.h): the extreme region pixels sit exactly on the rectangle's end edges
    double dx, dy;
    ddtrig::sincos_cr(theta, &dy, &dx);
    double l_min = 0, l_max = 0, w_min = 0, w_max = 0;           // max(0, max l), min(0, min l): order-independent
#pragma unroll 2
    for (int i = lane; i < n; i += 32) {                         // (no NaNs here: plain compares instead of fmax/fmin)
        const unsigned pk = reg[i];
        const double rdx = (double)(pk & 0xffff) - x, rdy = (double)(pk >> 16) - y;
        const double l = rdx * dx + rdy * dy, ww = -rdx * dy + rdy * dx;
        l_max = l > l_max ? l : l_max; l_min = l < l_min ? l : l_min; w_max = ww > w_max ? ww : w_max; w_min = ww < w_min ? ww : w_min;
    }
#pragma unroll 1
    for (int o = 16; o > 0; o >>= 1) {
        const double a = __shfl_xor_sync(0xffffffffu, l_max, o), b = __shfl_xor_sync(0xffffffffu, l_min, o);
        const double c = __shfl_xor_sync(0xffffffffu, w_max, o), d = __shfl_xor_sync(0xffffffffu, w_min, o);
        l_max = a > l_max ? a : l_max; l_min = b < l_min ? b : l_min; w_max = c > w_max ? c : w_max; w_min = d < w_min ? d : w_min;
    }
    LRect rec;
    rec.x1 = x + l_min * dx; rec.y1 = y + l_min * dy; rec.x2 = x + l_max * dx; rec.y2 = y + l_max * dy;
    rec.width = w_max - w_min; rec.x = x; rec.y = y; rec.theta = theta; rec.dx = dx; rec.dy = dy; rec.prec = prec; rec.p = p;
    if (rec.width < 1.0) rec.width = 1.0;
    *out = rec;
}

__device__ __forceinline__ double l_dist(double x1, double y1, double x2, double y2) { return sqrt((x2 - x1) * (x2 - x1) + (y2 - y1) * (y2 - y1)); }
__device__ __forceinline__ double l_distsq(double x1, double y1, double x2, double y2) { return (x2 - x1) * (x2 - x1) + (y2 - y1) * (y2 - y1); }

// reduce_region_radius (lsd.cpp).  The reference removes far points by swap-with-last while scanning forward, which
// leaves the kept points in a definite order (it matters: region2rect sums in list order): every kept point below the
// new size m' stays where it is, and the holes below m' (ascending) receive the kept points from positions >= m'
// in DESCENDING position order.  That is computed here chunk-wise with ballots: a descending cursor collects
// "fillers", an ascending one "holes", matched through a 32-entry shared buffer.  The removed tail's order is
// irrelevant (those points are only un-marked).
template <int SOLO> __device__ __noinline__ bool l_reduce_region_radius(int* n_io, double reg_angle, double prec, double p, LRect* rec, double density, double density_th) {
    const int lane = threadIdx.x & 31, w = s_W.w;
    int n = *n_io;
    if (SOLO == 0 && s_W.mode == 0) {  // speculative attempt: keep the list as it is (the commit validates every pixel ever accepted) and work on a copy
        if (2 * n + s_W.nasm > s_W.cap) { s_W.abort = 1; return false; }
        for (int i = lane; i < n; i += 32) s_W.reg[n + i] = s_W.reg[i];
        s_W.reg += n; s_W.cap -= n;
        __syncwarp();
    }
    unsigned* reg = s_W.reg;
    unsigned* s_fill = reinterpret_cast<unsigned*>(s_st);             // 32 filler values (s_st is free between region2rect calls)
    const unsigned p0 = reg[0];
    const double xc = (double)(p0 & 0xffff), yc = (double)(p0 >> 16);
    double radSq = fmax(l_distsq(xc, yc, rec->x1, rec->y1), l_distsq(xc, yc, rec->x2, rec->y2));
    while (density < density_th) {
        radSq *= 0.75 * 0.75;
        // pass 1: count the kept points, un-mark the removed ones
        int kept = 0;
#pragma unroll 1
        for (int b = 0; b < n; b += 32) {
            const int i = b + lane;
            bool keep = false;
            if (i < n) {
                const unsigned pk = reg[i];
                keep = !(l_distsq(xc, yc, (double)(pk & 0xffff), (double)(pk >> 16)) > radSq);
                if (!keep) l_release<SOLO>(s_W, (int)(pk >> 16) * w + (int)(pk & 0xffff));
            }
            kept += __popc(__ballot_sync(0xffffffffu, keep));
        }
        const int m2 = kept;
        // pass 2: fill the holes below m2 (ascending) with the kept points at or above m2 (descending)
        int lo = 0;                      // next hole chunk start (ascending, < m2)
        int hi = n;                      // filler cursor: positions [m2, hi) not yet consumed
        int nfill = 0, fpos = 0;         // fillers staged in s_fill[fpos .. nfill)
        while (lo < m2) {
            const int i = lo + lane;
            unsigned pk = 0; bool hole = false;
            if (i < m2) { pk = reg[i]; hole = l_distsq(xc, yc, (double)(pk & 0xffff), (double)(pk >> 16)) > radSq; }
            unsigned hm = __ballot_sync(0xffffffffu, hole);
            while (hm) {
                if (fpos == nfill) {     // stage the next (up to 32) fillers, descending from hi
                    nfill = 0; fpos = 0;
                    while (nfill == 0 && hi > m2) {
                        const int j = hi - 1 - lane;
                        unsigned fk = 0; bool isf = false;
                        if (j >= m2) { fk = reg[j]; isf = !(l_distsq(xc, yc, (double)(fk & 0xffff), (double)(fk >> 16)) > radSq); }
                        const unsigned fm = __ballot_sync(0xffffffffu, isf);
                        if (isf) s_fill[__popc(fm & ((1u << lane) - 1u))] = fk;
                        nfill = __popc(fm);
                        hi -= 32;
                    }
                    __syncwarp();
                    if (nfill == 0) break;                      // cannot happen (holes below m2 == kept at/above m2)
                }
                const int t = min(__popc(hm), nfill - fpos);    // holes served in this step
                const int r = __popc(hm & ((1u << lane) - 1u)); // this lane's rank among the pending holes
                if (((hm >> lane) & 1u) && r < t) reg[i] = s_fill[fpos + r];
                fpos += t;
                // drop the t lowest set bits of hm
                unsigned served = __ballot_sync(0xffffffffu, ((hm >> lane) & 1u) && r < t);
                hm &= ~served;
                __syncwarp();
            }
            lo += 32;
        }
        n = m2;
        __syncwarp();
        if (n < 2) { *n_io = n; return false; }
        l_region2rect<SOLO>(n, reg_angle, prec, p, rec);
        density = (double)n / (l_dist(rec->x1, rec->y1, rec->x2, rec->y2) * rec->width);
    }
    *n_io = n;
    return true;
}

template <int SOLO> __device__ __noinline__ bool l_refine(int* n_io, double* reg_angle_io, double prec, double p, LRect* rec, double density_th) {
    const int lane = threadIdx.x & 31, w = s_W.w;
    int n = *n_io;
    double density = (double)n / (l_dist(rec->x1, rec->y1, rec->x2, rec->y2) * rec->width);
    if (density >= density_th) return true;
    const unsigned* reg = s_W.reg; const float* __restrict__ ang = s_W.ang;
    const unsigned p0 = reg[0];
    const int sx = p0 & 0xffff, sy = p0 >> 16;
    const double xc = (double)sx, yc = (double)sy;
    const double ang_c = (double)ang[sy * w + sx] * L_DEG;
    const double width = rec->width;
    double* s0 = s_st; double* s1 = s_st + 32;
    const double* sp = s_st + (lane & 1) * 32;        // lane parity picks the accumulator: sum of d / sum of d*d
    double acc = 0; int cnt = 0;
#pragma unroll 1
    for (int b = 0; b < n; b += 32) {
        const int i = b + lane;
        bool in = false;
        if (i < n) {
            const unsigned pk = reg[i]; const int rx = pk & 0xffff, ry = pk >> 16;
            const float ad = ang[ry * w + rx];
            l_release<SOLO>(s_W, ry * w + rx);
            in = l_dist(xc, yc, (double)rx, (double)ry) < width;
            const double d = l_angle_diff_signed((double)ad * L_DEG, ang_c);
            // skipped points contribute +0.0, which leaves a running sum unchanged (the sums are never -0.0)
            s0[lane] = in ? d : 0.0; s1[lane] = in ? d * d : 0.0;
        }
        cnt += __popc(__ballot_sync(0xffffffffu, in));
        __syncwarp();
        acc = l_chunk_sum<SOLO>(sp, min(32, n - b), acc);
        __syncwarp();
    }
    const double sum = __shfl_sync(0xffffffffu, acc, 0), s_sum = __shfl_sync(0xffffffffu, acc, 1);
    const double mean_angle = sum / (double)cnt;
    const double tau = 2.0 * sqrt((s_sum - 2.0 * mean_angle * sum) / (double)cnt + mean_angle * mean_angle);
    __syncwarp();
    if (SOLO == 0 && s_W.mode == 0) { s_W.reg += n; s_W.cap -= n; }   // speculative: the first list stays (validated at commit), the regrown one follows it
    n = l_region_grow<SOLO>(sx, sy, tau, reg_angle_io);
    if (n < 0) { *n_io = 0; return false; }
    if (SOLO == 0 && s_W.mode == 0) s_W.acc += n;
    *n_io = n;
    if (n < 2) return false;
    l_region2rect<SOLO>(n, *reg_angle_io, prec, p, rec);
    density = (double)n / (l_dist(rec->x1, rec->y1, rec->x2, rec->y2) * rec->width);
    if (density < density_th) return l_reduce_region_radius<SOLO>(n_io, *reg_angle_io, prec, p, rec, density, density_th);
    return true;
}

__device__ double l_log_gamma(double x) {
    if (x > 15.0) return 0.918938533204673 + (x - 0.5) * log(x) - x + 0.5 * x * log(x * sinh(1 / x) + 1 / (810.0 * pow(x, 6.0)));
    const double q[7] = {75122.6331530, 80916.6278952, 36308.2951477, 8687.24529705, 1168.92649479, 83.8676043424, 2.50662827511};
    double a = (x + 0.5) * log(x + 5.5) - (x + 5.5), b = 0;
    for (int n = 0; n < 7; ++n) { a -= log(x + (double)n); b += q[n] * pow(x, (double)n); }
    return a + log(b);
}

__device__ __noinline__ double l_log(double x) { return log(x); }          // one copy of each libm routine per kernel
__device__ __noinline__ double l_log10(double x) { return log10(x); }
__device__ __noinline__ double l_exp(double x) { return exp(x); }
// (a real call everywhere: log / exp / pow / log10 inline to ~10 KB of SASS, and the NFA kernels keep thousands of
// warps at different program counters — code size is what their instruction cache sees)
__device__ __noinline__ double l_nfa(int n, int k, double p, double LOG_NT, const double* lgam) {
    if (n == 0 || k == 0) return -LOG_NT;
    if (n == k) return -LOG_NT - (double)n * l_log10(p);
    const double p_term = p / (1 - p);
    const double log1term = lgam[n] - lgam[k] - lgam[n - k] +
                            (double)k * l_log(p) + (double)(n - k) * l_log(1.0 - p);
    double term = l_exp(log1term);
    {   // double_equal(term, 0)
        bool eq = term == 0.0;
        if (!eq) { double abs_max = fabs(term); if (abs_max < 2.2250738585072014e-308) abs_max = 2.2250738585072014e-308; eq = (fabs(term) / abs_max) <= (100.0 * 2.220446049250313e-16); }
        if (eq) {
            if ((double)k > (double)n * p) return -log1term / 2.30258509299404568402 - LOG_NT;
            return -LOG_NT;
        }
    }
    double bin_tail = term;
    for (int i = k + 1; i <= n; i++) {
        const double bin_term = (double)(n - i + 1) / (double)i;
        const double mult_term = bin_term * p_term;
        term *= mult_term;
        bin_tail += term;
        if (bin_term < 1) {
            // pow(mult_term, m) < 2^-56 whenever mult_term < 1/4 and m >= 28; then 1 - pow rounds to exactly 1.0: skipping
            // the call is bit-identical (mult_term = bin_term * p / (1 - p) < 1/7 here for every p <= 1/8)
            const int m = n - i + 1;
            const double pw = (m >= 28 && mult_term < 0.25) ? 0.0 : pow(mult_term, (double)m);
            const double err = term * ((1 - pw) / (1 - mult_term) - 1);
            // threshold 0.1 * |-l_log10(bin_tail) - LOG_NT| * bin_tail: bracket log10 by the binary exponent first and
            // evaluate the logarithm only when the bracket cannot decide (same decision as the plain test, always)
            bool stop;
            const int e2 = ilogb(bin_tail);
            if (e2 > -1000 && e2 < 1000) {
                const double l_lo = -((double)(e2 + 1) * 0.30102999566398120) - LOG_NT, l_hi = -((double)e2 * 0.30102999566398120) - LOG_NT;  // L in [l_lo, l_hi]
                const double a_lo = (l_lo > 0) ? l_lo : ((l_hi < 0) ? -l_hi : 0.0), a_hi = fmax(fabs(l_lo), fabs(l_hi));
                if (err < 0.1 * a_lo * bin_tail * (1 - 1e-9)) stop = true;
                else if (err >= 0.1 * a_hi * bin_tail * (1 + 1e-9)) stop = false;
                else stop = err < 0.1 * fabs(-l_log10(bin_tail) - LOG_NT) * bin_tail;
            } else stop = err < 0.1 * fabs(-l_log10(bin_tail) - LOG_NT) * bin_tail;
            if (stop) break;
        }
    }
    return -l_log10(bin_tail) - LOG_NT;
}

__device__ __forceinline__ int l_x86_d2i(double v) {                 // cvttsd2si semantics
    if (!(v > -2147483649.0 && v < 2147483648.0)) return INT_MIN;
    return (int)v;
}

// rect_nfa of OpenCV 4.13 (see oracle/line_oracle.cpp): rows are distributed over the lanes (or, for flat
// rectangles, the pixels of a row); the two counts are exact integers, so the reduction order is irrelevant.
__device__ void l_rect_count(const Walk& W, const LRect& rec, int& total_out, int& alg_out) {
    const double half_width = 0.5 * rec.width, dyhw = rec.dy * half_width, dxhw = rec.dx * half_width;
    const double vx[4] = {rec.x1 - dyhw, rec.x2 - dyhw, rec.x2 + dyhw, rec.x1 + dyhw};
    const double vy[4] = {rec.y1 + dxhw, rec.y2 + dxhw, rec.y2 - dxhw, rec.y1 - dxhw};
    int off = 0;
#pragma unroll
    for (int i = 1; i < 4; i++) if (vy[i] < vy[off] || (vy[i] == vy[off] && vx[i] < vx[off])) off = i;
    const double Mx = vx[off], My = vy[off], Ax = vx[(off + 1) & 3], Ay = vy[(off + 1) & 3];
    const double Bx = vx[(off + 2) & 3], By = vy[(off + 2) & 3], Cx = vx[(off + 3) & 3], Cy = vy[(off + 3) & 3];
    const int cM = l_x86_d2i(ceil(My)), cA = l_x86_d2i(ceil(Ay)), cB = l_x86_d2i(ceil(By)), cC = l_x86_d2i(ceil(Cy));
    const double s1 = (cA != cM) ? (Ax - Mx) / (Ay - My) : 0.0;
    const double s2 = (cB != cA) ? (Bx - Ax) / (By - Ay) : 0.0;
    const double s3 = (cC != cM) ? (Cx - Mx) / (Cy - My) : 0.0;
    const double s4 = (cB != cC) ? (Bx - Cx) / (By - Cy) : 0.0;
    int total = 0, alg = 0;
    const int y0 = max(cM, 0), y1 = min(cB, W.h - 1);
    const bool by_rows = (y1 - y0) >= 16;
    for (int yb = y0; yb <= y1; yb += by_rows ? 32 : 1) {
        const int y = by_rows ? yb + W.lane : yb;
        if (y > y1) continue;
        const double xl = (cA < y) ? ((double)y - Ay) * s2 + Ax : ((double)y - My) * s1 + Mx;
        const double xr = (cC <= y) ? ((double)y - Cy) * s4 + Cx : ((double)y - My) * s3 + Mx;
        int xs = l_x86_d2i(ceil(xl));
        int xe = l_x86_d2i(xr);
        if (xe < xs) continue;
        if (xs < 0) xs = 0;
        if (xe > W.w - 1) xe = W.w - 1;
        const float* row = W.ang + (long long)y * W.w;
        if (by_rows) {
            for (int x = xs; x <= xe; ++x) { ++total; if (l_aligned(row[x], rec.theta, rec.prec)) ++alg; }
        } else {
            for (int x = xs + W.lane; x <= xe; x += 32) { ++total; if (l_aligned(row[x], rec.theta, rec.prec)) ++alg; }
        }
    }
    total_out = __reduce_add_sync(0xffffffffu, total);
    alg_out = __reduce_add_sync(0xffffffffu, alg);
}

__device__ double l_rect_nfa(const Walk& W, const LRect& rec) {
    int total, alg;
    l_rect_count(W, rec, total, alg);
    return l_nfa(total, alg, rec.p, W.log_nt, W.lgam);
}

// Five candidate rectangles of one rect_improve phase at once: lane group g = lane / 6 (6 lanes each, lanes 30-31 idle)
// scans candidate g's rows, the counts are combined through shared-memory atomics (exact integers), and the five
// scalar NFA evaluations run side by side in lanes 0, 6, 12, 18, 24.  s_cnt: 10 ints of this warp.
__device__ __noinline__ void l_rect_nfa5(const Walk& W, const LRect& mine, bool valid, int* s_cnt, double* out5) {
    const int lane = W.lane, grp = lane / 6, sub = lane - grp * 6;
    if (lane < 10) s_cnt[lane] = 0;
    __syncwarp();
    if (grp < 5 && valid) {
        const LRect& rec = mine;
        const double half_width = 0.5 * rec.width, dyhw = rec.dy * half_width, dxhw = rec.dx * half_width;
        const double vx[4] = {rec.x1 - dyhw, rec.x2 - dyhw, rec.x2 + dyhw, rec.x1 + dyhw};
        const double vy[4] = {rec.y1 + dxhw, rec.y2 + dxhw, rec.y2 - dxhw, rec.y1 - dxhw};
        int off = 0;
#pragma unroll
        for (int i = 1; i < 4; i++) if (vy[i] < vy[off] || (vy[i] == vy[off] && vx[i] < vx[off])) off = i;
        const double Mx = vx[off], My = vy[off], Ax = vx[(off + 1) & 3], Ay = vy[(off + 1) & 3];
        const double Bx = vx[(off + 2) & 3], By = vy[(off + 2) & 3], Cx = vx[(off + 3) & 3], Cy = vy[(off + 3) & 3];
        const int cM = l_x86_d2i(ceil(My)), cA = l_x86_d2i(ceil(Ay)), cB = l_x86_d2i(ceil(By)), cC = l_x86_d2i(ceil(Cy));
        const double s1 = (cA != cM) ? (Ax - Mx) / (Ay - My) : 0.0;
        const double s2 = (cB != cA) ? (Bx - Ax) / (By - Ay) : 0.0;
        const double s3 = (cC != cM) ? (Cx - Mx) / (Cy - My) : 0.0;
        const double s4 = (cB != cC) ? (Bx - Cx) / (By - Cy) : 0.0;
        int total = 0, alg = 0;
        const int y0 = max(cM, 0), y1 = min(cB, W.h - 1);
        for (int y = y0 + sub; y <= y1; y += 6) {
            const double xl = (cA < y) ? ((double)y - Ay) * s2 + Ax : ((double)y - My) * s1 + Mx;
            const double xr = (cC <= y) ? ((double)y - Cy) * s4 + Cx : ((double)y - My) * s3 + Mx;
            int xs = l_x86_d2i(ceil(xl));
            int xe = l_x86_d2i(xr);
            if (xe < xs) continue;
            if (xs < 0) xs = 0;
            if (xe > W.w - 1) xe = W.w - 1;
            const float* row = W.ang + (long long)y * W.w;
            for (int x = xs; x <= xe; ++x) { ++total; if (l_aligned(__ldg(row + x), rec.theta, rec.prec)) ++alg; }
        }
        if (total) atomicAdd(&s_cnt[2 * grp], total);
        if (alg) atomicAdd(&s_cnt[2 * grp + 1], alg);
    }
    __syncwarp();
    double v = 0.0;
    if (grp < 5 && sub == 0 && valid) v = l_nfa(s_cnt[2 * grp], s_cnt[2 * grp + 1], mine.p, W.log_nt, W.lgam);
#pragma unroll
    for (int g5 = 0; g5 < 5; g5++) out5[g5] = __shfl_sync(0xffffffffu, v, g5 * 6);
    __syncwarp();
}

// rect_improve (lsd.cpp): each of the five refinement phases tries a fixed sequence of five candidate rectangles that
// does not depend on the NFA values inside the phase, so the five are evaluated at once (l_rect_nfa5) and the
// reference's "first strict improvement wins" rule is then replayed in order.
__device__ double l_rect_improve(const Walk& W, LRect& rec, int* s_cnt, double log_nfa) {
    const double delta = 0.5, delta_2 = delta / 2.0;
    const int lane = W.lane, grp = lane / 6, k = min(grp, 4) + 1;     // this lane's candidate = k-th step of the phase
    if (log_nfa > 0.0) return log_nfa;           // log_nfa = NFA of the unmodified rectangle (k_lsd_nfa_first)
    double v[5];
#pragma unroll 1
    for (int phase = 0; phase < 5; phase++) {
        // candidate k of the phase, built exactly as the sequential loop would have built it
        LRect r = rec;
        bool valid = true;
        if (phase == 0 || phase == 4) {
            if (phase == 4) valid = (r.width - delta) >= 0.5;          // the guard does not change inside the loop
            for (int i = 0; i < k; i++) { r.p /= 2; r.prec = r.p * L_PI; }
        } else {
            for (int i = 0; i < k; i++) {
                if ((r.width - delta) >= 0.5) {
                    if (phase == 2) { r.x1 += -r.dy * delta_2; r.y1 += r.dx * delta_2; r.x2 += -r.dy * delta_2; r.y2 += r.dx * delta_2; }
                    if (phase == 3) { r.x1 -= -r.dy * delta_2; r.y1 -= r.dx * delta_2; r.x2 -= -r.dy * delta_2; r.y2 -= r.dx * delta_2; }
                    r.width -= delta;
                } else valid = false;                                   // this step (and all later ones) is skipped
            }
        }
        l_rect_nfa5(W, r, valid, s_cnt, v);
        // replay: for n = 1..5: if (candidate n exists && v_n > log_nfa) { log_nfa = v_n; rec = candidate n; }
        int best = -1;
        for (int n = 0; n < 5; n++) {
            const bool vn = __shfl_sync(0xffffffffu, valid ? 1 : 0, n * 6) != 0;
            if (vn && v[n] > log_nfa) { log_nfa = v[n]; best = n; }
        }
        if (best >= 0) {                                                // broadcast the winning candidate's fields
            const int src = best * 6;
            rec.x1 = __shfl_sync(0xffffffffu, r.x1, src); rec.y1 = __shfl_sync(0xffffffffu, r.y1, src);
            rec.x2 = __shfl_sync(0xffffffffu, r.x2, src); rec.y2 = __shfl_sync(0xffffffffu, r.y2, src);
            rec.width = __shfl_sync(0xffffffffu, r.width, src);
            rec.p = __shfl_sync(0xffffffffu, r.p, src); rec.prec = __shfl_sync(0xffffffffu, r.prec, src);
        }
        if (log_nfa > 0.0) return log_nfa;
    }
    return log_nfa;
}

// The order-dependent core: seeds in order, region growing, rectangle fit and the density refinement (the only steps
// that read or write the `used` map).  rect_improve / NFA of a region is a pure function of its rectangle and of the
// immutable angle map, so it is NOT done here: the walker emits one job per candidate region and k_lsd_nfa evaluates
// all jobs of all frames in parallel (one warp per job).
//
// ONE CTA PER FRAME, several warps, exact sequential semantics.  The regions of a frame form a sparse dependency graph
// (tools/sim_spec_walker.cpp: critical path 1/17 of the work at 640x480, 1/100 at 1280x960), but which regions exist and
// what they depend on is only known by running them.  So the warps run region growing AHEAD of the sequential order and
// the results are committed strictly IN that order:
//   * claim  (claim_lock, shared memory only): the next seed, in seed order, that is not in the committed bitmap gets the
//     next rank `seq` and a slot of a ring (its own list buffer);
//   * attempt (any warp, speculative): grow / fit / refine exactly as the sequential code would, reading "used" as
//     committed bitmap | my ticket | live ticket of lower rank (the last one recorded as an assumption), writing only
//     tickets (LPix.used, global) and its private lists.  A seed already under a live ticket of lower rank is presumed
//     swallowed; an attempt that loses a pixel to a live attempt of lower rank waits for that rank to retire and starts over;
//   * commit (commit_lock, in rank order, by whichever warp is idle): the attempt is VALID iff it was not poisoned, none
//     of the pixels it ever accepted is in the committed bitmap and all the pixels it assumed used are.  Then every
//     membership test it made had the sequential outcome, so its lists are the sequential ones: its final pixels are
//     published to the bitmap and its job appended.  Otherwise (and for presumed seeds that were not swallowed after all)
//     the region is grown on the spot by the "turn holder": everything of lower rank is final, nothing can invalidate it.
// Bits only go 0 -> 1 and are written only under commit_lock; tickets of retired ranks are garbage by construction.
__device__ __forceinline__ void l_unlock(int* l) { __threadfence_block(); atomicExch(l, 0); }

struct WalkFrame { const LineGeom* g; const LineWs* ws; int f; unsigned* bits; };

// grow + fit + refine one seed.  Returns 1 = candidate rectangle in *rec, 0 = no job (small or rejected by refine), -1 = abandoned.
// *n0 = size of the first region, *nfin = pixels that stay used (the list at s_W.reg).
__device__ __noinline__ int l_one_region(const LineGeom& g, unsigned idx, LRect* rec, int* n0, int* nfin) {
    WalkCtx& W = s_W;
    double reg_angle;
    int n = l_region_grow<0>((int)(idx % (unsigned)g.sw), (int)(idx / (unsigned)g.sw), g.prec, &reg_angle);
    if (n < 0) return -1;
    W.acc = n;
    *n0 = n; *nfin = n;
    if (n < g.min_reg_size) return 0;
    l_region2rect<0>(n, reg_angle, g.prec, g.p, rec);
    const bool okr = l_refine<0>(&n, &reg_angle, g.prec, g.p, rec, 0.7);
    if (W.abort) return -1;
    *nfin = n;
    return okr ? 1 : 0;
}

__device__ __forceinline__ void l_emit_job(const LineGeom& g, double* dst, const LRect& rec, unsigned idx, int n0, int lane) {
    if (lane < 13) {
        const double v[13] = {rec.x1, rec.y1, rec.x2, rec.y2, rec.width, rec.x, rec.y, rec.theta, rec.dx, rec.dy, rec.prec, rec.p, (double)idx * 65536.0 + (double)min(n0, 65535)};
        double out = v[0];
#pragma unroll
        for (int k = 1; k < 13; k++) if (lane == k) out = v[k];
        dst[lane] = out;
    }
}

__device__ __forceinline__ void l_set_bit(unsigned* bits, unsigned pk, int w) { const int q = (int)(pk >> 16) * w + (int)(pk & 0xffff); atomicOr(bits + (q >> 5), 1u << (q & 31)); }

// The turn holder grows the region of seed `idx` for real (commit_lock held, every lower rank committed).
__device__ __noinline__ void l_turn_region(const WalkFrame& F, unsigned idx, int seq) {
    const LineGeom& g = *F.g; const LineWs& ws = *F.ws;
    const int lane = threadIdx.x & 31;
    const long long t0 = clock64();
    WalkCtx& W = s_W;
    __syncwarp();
    if (lane == 0) {
        W.mode = 1; W.abort = 0; W.seq = seq; W.ticket = (unsigned)(seq + 1) | 0x80000000u;
        W.reg = ws.reg + (long long)F.f * g.pix_stride; W.base0 = W.reg; W.cap = (int)g.pix_stride; W.nasm = 0; W.acc = 0;
    }
    __syncwarp();
    LRect rec; int n0 = 0, nfin = 0;
    const int r = l_one_region(g, idx, &rec, &n0, &nfin);
    __syncwarp();
    for (int i = lane; i < nfin; i += 32) l_set_bit(F.bits, W.reg[i], g.sw);
    if (r == 1) {
        const int nj = s_F.nj;
        if (nj < g.seg_cap) l_emit_job(g, ws.jobs + ((long long)F.f * g.seg_cap + nj) * 13, rec, idx, n0, lane);
        __syncwarp();
        if (lane == 0) s_F.nj = nj + 1;
    }
    __syncwarp();
    if (lane == 0 && (g.dbg & 32)) { atomicAdd(ws.wstat + 0, 1ull); atomicAdd(ws.wstat + 1, (unsigned long long)(clock64() - t0)); atomicAdd(ws.wstat + 2, (unsigned long long)nfin); }
}

// commit slot `k` (rank `seq`); commit_lock held
__device__ __noinline__ void l_commit_slot(const WalkFrame& F, int k, int seq) {
    const LineGeom& g = *F.g; const LineWs& ws = *F.ws;
    const int lane = threadIdx.x & 31;
    const int st = s_F.state[k];
    if (s_F.seedpix[k] < 0) return;                               // the sentinel claim that closes the frame
    const unsigned idx = (unsigned)s_F.seedpix[k];
    if (l_bit(F.bits, (int)idx)) { if (lane == 0 && (g.dbg & 32)) atomicAdd(ws.wstat + 4, 1ull); return; }     // swallowed by a region of lower rank: nothing to do
    bool ok = st == SLOT_DONE && !s_F.poison[k];
    const int acc = s_F.acc[k], nasm = s_F.nasm[k], finoff = s_F.finoff[k], nfin = s_F.nfin[k];
    const bool small = finoff == 0 && acc + nasm <= WALK_SMALL && !(g.dbg & 2);    // everything needed is in shared memory
    const unsigned* list = ws.sreg + ((long long)F.f * WALK_RING + k) * WALK_SLOT_CAP;
    if (ok) {
        bool bad = false;
        if (small) {
            if (lane < acc) { const unsigned pk = s_F.small[k][lane]; bad = l_bit(F.bits, (int)(pk >> 16) * g.sw + (int)(pk & 0xffff)); }
            else if (lane < acc + nasm) bad = !l_bit(F.bits, (int)s_F.small[k][lane]);
        } else {
            for (int i = lane; i < acc; i += 32) { const unsigned pk = __ldcg(list + i); bad |= l_bit(F.bits, (int)(pk >> 16) * g.sw + (int)(pk & 0xffff)); }
            for (int i = lane; i < nasm; i += 32) bad |= !l_bit(F.bits, (int)__ldcg(list + WALK_SLOT_CAP - 1 - i));
        }
        ok = !__any_sync(0xffffffffu, bad);
    }
    if (!ok) {
        if (lane == 0 && (g.dbg & 32)) atomicAdd(ws.wstat + 5 + (st == SLOT_PRESUMED ? 3 : (st != SLOT_DONE ? 0 : (s_F.poison[k] ? 1 : 2))), 1ull);
        l_turn_region(F, idx, seq);
        return;
    }
    if (lane == 0 && (g.dbg & 32)) { atomicAdd(ws.wstat + 9, 1ull); atomicAdd(ws.wstat + 10, (unsigned long long)nfin); }
    if (small) { if (lane < nfin) l_set_bit(F.bits, s_F.small[k][lane], g.sw); }
    else for (int i = lane; i < nfin; i += 32) l_set_bit(F.bits, __ldcg(list + finoff + i), g.sw);
    if (s_F.job[k]) {
        const int nj = s_F.nj;
        if (nj < g.seg_cap && lane < 13) ws.jobs[((long long)F.f * g.seg_cap + nj) * 13 + lane] = s_F.jobv[k][lane];
        __syncwarp();
        if (lane == 0) s_F.nj = nj + 1;
    }
    __syncwarp();
}

// claim the next seed (claim_lock held by this warp): returns the slot, -1 when the ring is full, -2 for the closing sentinel
__device__ __noinline__ int l_claim(const WalkFrame& F) {
    const LineGeom& g = *F.g; const LineWs& ws = *F.ws;
    const int lane = threadIdx.x & 31;
    const unsigned* seeds = ws.seeds + (long long)F.f * g.pix_stride;
    const int ns = s_F.ns;
    const unsigned nclaims = s_F.nclaims;
    if (s_F.all_claimed || nclaims - l_turn() >= (unsigned)WALK_RING) return -1;
    const int k = (int)(nclaims % WALK_RING);
    if (*reinterpret_cast<volatile int*>(&s_F.state[k]) != SLOT_EMPTY) return -1;
    int cur = (int)s_F.cursor, found = ns;
    unsigned pixidx = 0;
    while (cur < ns) {
        int wb = s_F.win_base;
        if (cur < wb || cur >= wb + WALK_WIN) {                    // stage the next window of the ordered seed list
            wb = cur & ~31;
            for (int i = lane; i < WALK_WIN; i += 32) s_F.win[i] = wb + i < ns ? seeds[wb + i] : 0u;
            if (lane == 0) s_F.win_base = wb;
            __syncwarp();
        }
        const int i = cur + lane;
        const bool have = i < ns && i < wb + WALK_WIN;
        const unsigned mine = have ? s_F.win[i - wb] : 0u;
        const unsigned fm = __ballot_sync(0xffffffffu, have && !l_bit(F.bits, (int)mine));
        if (fm) { const int j = __ffs(fm) - 1; found = cur + j; pixidx = __shfl_sync(0xffffffffu, mine, j); break; }
        cur = min(cur + 32, wb + WALK_WIN);
    }
    if (lane == 0) {
        s_F.seqof[k] = (int)nclaims; s_F.seedpix[k] = found >= ns ? -1 : (int)pixidx; s_F.poison[k] = 0; s_F.job[k] = 0;
        *reinterpret_cast<volatile int*>(&s_F.state[k]) = found >= ns ? SLOT_ABORTED : SLOT_RUNNING;     // the sentinel has nothing to grow
        s_F.cursor = (unsigned)min(found + 1, ns);
        if (found >= ns) s_F.all_claimed = 1;
        __threadfence_block();
        s_F.nclaims = nclaims + 1;
    }
    __syncwarp();
    return found >= ns ? -2 : k;
}

// 128 registers: a build held to 80 (three 8-warp CTAs per SM) spilled and was 15-20 % slower in every configuration measured
__global__ void __launch_bounds__(WALK_MAXW * 32) k_lsd_regions(const __grid_constant__ LineGeom g, LineWs ws, int nframes) {
    extern __shared__ unsigned s_bits[];                       // committed `used` bitmap of the frame
    const int lane = threadIdx.x & 31;
    const int nwords = (int)((g.pix_stride + 31) >> 5);
  for (;;) {
    // frames are pulled from a counter: the grid may be smaller than the batch (sslpl_line_set_max_walkers)
    __syncthreads();
    if (threadIdx.x == 0) {
        const int f = atomicAdd(ws.rejctl + 2, 1);
        s_F.frame = f; s_F.cursor = 0; s_F.nclaims = 0; s_F.turn = 0; s_F.claim_lock = 0; s_F.commit_lock = 0; s_F.all_claimed = 0; s_F.nj = 0; s_F.win_base = -(1 << 30);
        s_F.ns = f < nframes ? ws.nseeds[f] : 0;
        for (int k = 0; k < WALK_RING; k++) { s_F.state[k] = SLOT_EMPTY; s_F.poison[k] = 0; }
    }
    for (int i = threadIdx.x; i < nwords; i += blockDim.x) s_bits[i] = 0u;
    __syncthreads();
    const int f = s_F.frame;
    if (f >= nframes) break;
    const long long tf0 = clock64();
    WalkFrame F; F.g = &g; F.ws = &ws; F.f = f; F.bits = s_bits;
    WalkCtx& W = s_W;
    if (lane == 0) {
        W.w = g.sw; W.h = g.sh;
        W.ang = ws.angdeg + f * g.pix_stride; W.mod = ws.modgrad + f * g.pix_stride;
        W.pix = ws.pix + f * g.pix_stride; W.cs0 = ws.cs0 + f * g.pix_stride; W.bits = s_bits; W.dbg = g.dbg;
    }
    __syncwarp();
    int myslot = -1, tries = 0, waitfor = -1;                  // an attempt of this warp waiting for rank `waitfor` to retire
    for (;;) {
        // ---- 1. commits, by whoever finds the head of the ring finished
        int did = 0;
        {
            int go = 0;
            if (lane == 0) {
                const unsigned t = l_turn();
                if (t < *reinterpret_cast<volatile unsigned*>(&s_F.nclaims)) {
                    const int st = *reinterpret_cast<volatile int*>(&s_F.state[t % WALK_RING]);
                    if (st >= SLOT_DONE && atomicCAS(&s_F.commit_lock, 0, 1) == 0) { __threadfence_block(); go = 1; }
                }
            }
            go = __shfl_sync(0xffffffffu, go, 0);
            if (go) {
                const long long tc0 = clock64();
                for (;;) {
                    const unsigned t = l_turn();
                    if (t >= *reinterpret_cast<volatile unsigned*>(&s_F.nclaims)) break;
                    const int k = (int)(t % WALK_RING);
                    if (*reinterpret_cast<volatile int*>(&s_F.state[k]) < SLOT_DONE) break;
                    __syncwarp();
                    l_commit_slot(F, k, (int)t);
                    __syncwarp();
                    if (lane == 0) { __threadfence_block(); *reinterpret_cast<volatile int*>(&s_F.state[k]) = SLOT_EMPTY; __threadfence_block(); *reinterpret_cast<volatile unsigned*>(&s_F.turn) = t + 1; }
                    __syncwarp();
                    did = 1;
                }
                if (lane == 0) { if (g.dbg & 32) atomicAdd(ws.wstat + 11, (unsigned long long)(clock64() - tc0)); l_unlock(&s_F.commit_lock); }
                __syncwarp();
            }
        }
        if (did) continue;
        // ---- 2. an attempt: a new claim, or the repetition of one that had to wait for a lower rank
        if (myslot < 0) {
            int go = 0;
            if (lane == 0 && !*reinterpret_cast<volatile int*>(&s_F.all_claimed) &&
                *reinterpret_cast<volatile unsigned*>(&s_F.nclaims) - l_turn() < (unsigned)WALK_RING && atomicCAS(&s_F.claim_lock, 0, 1) == 0) { __threadfence_block(); go = 1; }
            go = __shfl_sync(0xffffffffu, go, 0);
            if (go) {
                const long long tk0 = clock64();
                const int k = l_claim(F);
                if (lane == 0) { if (g.dbg & 32) atomicAdd(ws.wstat + 12, (unsigned long long)(clock64() - tk0)); l_unlock(&s_F.claim_lock); }
                __syncwarp();
                if (k >= 0) { myslot = k; tries = 0; waitfor = -1; }
            }
        }
        if (myslot >= 0 && (waitfor < 0 || (int)l_turn() > waitfor)) {
            const int k = myslot;
            const unsigned idx = (unsigned)s_F.seedpix[k];
            if (lane == 0) {
                W.mode = 0; W.abort = 0; W.conflict = -1; W.nasm = 0; W.acc = 0; W.seq = s_F.seqof[k];
                W.ticket = (unsigned)(W.seq + 1) | ((unsigned)(tries & 127) << 24);
                W.reg = ws.sreg + ((long long)f * WALK_RING + k) * WALK_SLOT_CAP; W.base0 = W.reg; W.cap = WALK_SLOT_CAP;
            }
            __syncwarp();
            LRect rec; int n0 = 0, nfin = 0;
            int r = -1;
            if (l_bit(s_bits, (int)idx)) { if (lane == 0) W.abort = 3; __syncwarp(); }     // swallowed while this attempt waited
            else r = l_one_region(g, idx, &rec, &n0, &nfin);
            __syncwarp();
            if (r < 0 && W.abort == 2 && tries < 100 && !(g.dbg & 1)) {           // a live attempt of lower rank holds a pixel this one needs: repeat after it retires
                waitfor = W.conflict; tries++;
                if (lane == 0 && (g.dbg & 32)) atomicAdd(ws.wstat + 13, 1ull);
                __syncwarp();
                continue;
            }
            if (r == 1) l_emit_job(g, s_F.jobv[k], rec, idx, n0, lane);
            int st = SLOT_DONE;
            if (r < 0) st = W.abort == 3 ? SLOT_PRESUMED : SLOT_ABORTED;
            else {
                const int acc = W.acc, nasm = W.nasm, finoff = (int)(W.reg - W.base0);
                if (finoff == 0 && acc + nasm <= WALK_SMALL && !(g.dbg & 2)) {   // small attempt: its lists travel through shared memory
                    if (lane < acc) s_F.small[k][lane] = W.base0[lane];
                    else if (lane < acc + nasm) s_F.small[k][lane] = W.base0[WALK_SLOT_CAP - 1 - (lane - acc)];
                }
                if (lane == 0) { s_F.acc[k] = acc; s_F.nasm[k] = nasm; s_F.finoff[k] = finoff; s_F.nfin[k] = nfin; s_F.job[k] = r == 1; }
            }
            __syncwarp();
            if (lane == 0) { __threadfence(); *reinterpret_cast<volatile int*>(&s_F.state[k]) = st; }
            __syncwarp();
            myslot = -1;
            continue;
        }
        // ---- 3. done?
        if (myslot < 0 && *reinterpret_cast<volatile int*>(&s_F.all_claimed) && l_turn() >= *reinterpret_cast<volatile unsigned*>(&s_F.nclaims)) break;
        __nanosleep(100);
    }
    __syncthreads();
    if (threadIdx.x == 0) { if (g.dbg & 32) { atomicAdd(ws.wstat + 14, (unsigned long long)(clock64() - tf0)); atomicAdd(ws.wstat + 15, (unsigned long long)s_F.nclaims); }
        ws.njobs[f] = min(s_F.nj, g.seg_cap); if (s_F.nj > g.seg_cap) atomicOr(ws.err, DERR_LSD_OVERFLOW); }
  }
}

// THROUGHPUT form of the same stage for big batches: ONE WARP PER FRAME, no speculation (every instruction is useful work, 72
// registers, ~28 frames resident per SM; 46 ms latency per frame, ~17 us per frame amortised with >= 3000 frames in flight).
// sslpl picks it when a call brings at least two frames per SM; smaller calls use the multi-warp walker above (17 ms per frame).
#ifndef SSLPL_SOLO_MINB
#define SSLPL_SOLO_MINB 28
#endif
__global__ void __launch_bounds__(32, SSLPL_SOLO_MINB) k_lsd_regions_solo(const __grid_constant__ LineGeom g, LineWs ws, int nframes) {
    const int lane = threadIdx.x;
  for (;;) {
    int f = 0;
    if (lane == 0) f = atomicAdd(ws.rejctl + 2, 1);
    f = __shfl_sync(0xffffffffu, f, 0);
    if (f >= nframes) break;
    __syncwarp();
    WalkCtx& W = s_W1;
    if (lane == 0) {
        W.w = g.sw; W.h = g.sh; W.mode = 2; W.abort = 0; W.nasm = 0; W.acc = 0; W.cap = (int)g.pix_stride; W.ticket = 1u; W.seq = 0;
        W.ang = ws.angdeg + f * g.pix_stride; W.mod = ws.modgrad + f * g.pix_stride;
        W.pix = ws.pix + f * g.pix_stride; W.reg = ws.reg + f * g.pix_stride; W.base0 = W.reg; W.cs0 = ws.cs0 + f * g.pix_stride; W.bits = nullptr;
    }
    __syncwarp();
    const LPix* pix = ws.pix + f * g.pix_stride;
    const unsigned* seeds = ws.seeds + f * g.pix_stride;
    const int ns = ws.nseeds[f];
    double* jobs = ws.jobs + (long long)f * g.seg_cap * 13;
    int nj = 0;
    for (int sb = 0; sb < ns; sb += 32) {
        const bool have = sb + lane < ns;
        const unsigned mine = have ? seeds[sb + lane] : 0u;                   // 32 seeds per coalesced load
        unsigned umask = __ballot_sync(0xffffffffu, !have || pix[mine].used != 0u); // their `used` state, one round trip
        while (~umask) {                                    // angle != NOTDEF holds for every seed
            const int j = __ffs(~umask) - 1;
            umask |= (2u << j) - 1u;                        // seeds up to j are done
            const unsigned idx = __shfl_sync(0xffffffffu, mine, j);
            double reg_angle;
            int n = l_region_grow<1>((int)(idx % (unsigned)g.sw), (int)(idx / (unsigned)g.sw), g.prec, &reg_angle);
            umask |= __ballot_sync(0xffffffffu, !have || pix[mine].used != 0u);    // the region may have swallowed later seeds
            if (n < g.min_reg_size) continue;
            LRect rec;
            l_region2rect<1>(n, reg_angle, g.prec, g.p, &rec);
            const int n0 = n;
            const bool okr = l_refine<1>(&n, &reg_angle, g.prec, g.p, &rec, 0.7);
            umask = ((2u << j) - 1u) | __ballot_sync(0xffffffffu, !have || pix[mine].used != 0u);   // refine can release and re-take pixels
            if (!okr) continue;
            if (nj < g.seg_cap) l_emit_job(g, jobs + (long long)nj * 13, rec, idx, n0, lane);
            nj++;
        }
    }
    if (lane == 0) { ws.njobs[f] = min(nj, g.seg_cap); if (nj > g.seg_cap) atomicOr(ws.err, DERR_LSD_OVERFLOW); }
    __syncwarp();
  }
}

// NFA of every candidate region of every frame, in three data-parallel steps (grids are sized by the work, not by the
// per-frame capacity seg_cap, which is ~13k slots of which a few hundred are used):
//   k_lsd_nfa_count   one warp per job: the rectangle scan (total / aligned pixel counts)
//   k_lsd_nfa_first   one THREAD per job: the scalar NFA formula (32 jobs per warp side by side); most jobs are accepted
//                     here, the others are appended to a global work list
//   k_lsd_nfa_improve persistent warps pull rejected jobs from that list: the five refinement phases of rect_improve
constexpr int NFA_COUNT_CTAS = 16;          // CTAs (4 warps) per frame in k_lsd_nfa_count
constexpr int NFA_FIRST_CTAS = 2;           // CTAs (128 threads) per frame in k_lsd_nfa_first

__device__ __forceinline__ void l_trace_row(const LineGeom& g, const LineWs& ws, int f, int j, const double* job, double tag, double log_nfa) {
    if (g.trace_cap && j < g.trace_cap) {
        double* t = ws.trace + ((long long)f * g.trace_cap + j) * 10;
        const double idx = floor(tag / 65536.0);
        t[0] = idx; t[1] = tag - idx * 65536.0; t[2] = 0; t[3] = log_nfa;
        t[4] = job[0]; t[5] = job[1]; t[6] = job[2]; t[7] = job[3]; t[8] = job[4]; t[9] = job[11];
    }
}

__global__ void __launch_bounds__(128) k_lsd_nfa_count(const __grid_constant__ LineGeom g, LineWs ws) {
    const int f = blockIdx.y, nj = ws.njobs[f];
    Walk W;
    W.w = g.sw; W.h = g.sh; W.lane = threadIdx.x & 31; W.ang = ws.angdeg + f * g.pix_stride; W.log_nt = g.log_nt; W.lgam = ws.lgam;
    for (int j = blockIdx.x * 4 + (threadIdx.x >> 5); j < nj; j += NFA_COUNT_CTAS * 4) {
        const double* job = ws.jobs + ((long long)f * g.seg_cap + j) * 13;
        LRect rec;
        rec.x1 = job[0]; rec.y1 = job[1]; rec.x2 = job[2]; rec.y2 = job[3]; rec.width = job[4]; rec.theta = job[7]; rec.dx = job[8]; rec.dy = job[9]; rec.prec = job[10];
        int total, alg;
        l_rect_count(W, rec, total, alg);
        if (W.lane == 0) ws.jobnk[(long long)f * g.seg_cap + j] = make_int2(total, alg);
    }
}

__global__ void __launch_bounds__(128) k_lsd_nfa_first(const __grid_constant__ LineGeom g, LineWs ws) {
    const int f = blockIdx.y, nj = ws.njobs[f];
    for (int j = blockIdx.x * 128 + threadIdx.x; j < nj; j += NFA_FIRST_CTAS * 128) {
        const long long q = (long long)f * g.seg_cap + j;
        const int2 nk = ws.jobnk[q];
        double* job = ws.jobs + q * 13;
        const double v = l_nfa(nk.x, nk.y, job[11], g.log_nt, ws.lgam);
        if (v > 0.0) {
            const double tag = job[12];
            ws.jobflag[q] = 1; job[12] = v;
            l_trace_row(g, ws, f, j, job, tag, v);
        } else {
            ws.jobflag[q] = 0; ws.jobnfa[q] = v;
            ws.rej[atomicAdd(ws.rejctl, 1)] = make_int2(f, j);     // order is irrelevant: results go back to the job slot
        }
    }
}

__global__ void __launch_bounds__(128) k_lsd_nfa_improve(const __grid_constant__ LineGeom g, LineWs ws) {
    __shared__ int s_cnt[4][10];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int nrej = ws.rejctl[0];
    for (;;) {
        int r = 0;
        if (lane == 0) r = atomicAdd(ws.rejctl + 1, 1);
        r = __shfl_sync(0xffffffffu, r, 0);
        if (r >= nrej) break;
        const int2 fj = ws.rej[r];
        const int f = fj.x, j = fj.y;
        const long long q = (long long)f * g.seg_cap + j;
        double log_nfa = ws.jobnfa[q];
        double* job = ws.jobs + q * 13;
        Walk W;
        W.w = g.sw; W.h = g.sh; W.lane = lane;
        W.ang = ws.angdeg + f * g.pix_stride; W.log_nt = g.log_nt; W.lgam = ws.lgam;
        LRect rec;
        rec.x1 = job[0]; rec.y1 = job[1]; rec.x2 = job[2]; rec.y2 = job[3]; rec.width = job[4]; rec.x = job[5]; rec.y = job[6];
        rec.theta = job[7]; rec.dx = job[8]; rec.dy = job[9]; rec.prec = job[10]; rec.p = job[11];
        const double tag = job[12];
        __syncwarp();
        log_nfa = l_rect_improve(W, rec, s_cnt[wid], log_nfa);
        __syncwarp();
        if (lane == 0) {
            job[0] = rec.x1; job[1] = rec.y1; job[2] = rec.x2; job[3] = rec.y2; job[4] = rec.width; job[11] = rec.p;
            ws.jobflag[q] = log_nfa > 0.0 ? 1 : 0;
            job[12] = log_nfa;
            l_trace_row(g, ws, f, j, job, tag, log_nfa);
        }
        __syncwarp();
    }
}

// cv::LineIterator(img, p1, p2, 8).count: the endpoints are cvRound()ed floats from [0, lim), so 639.6 becomes 640 — one past
// the last column — and OpenCV clips the segment to the image (cv::clipLine, 64-bit integer arithmetic) before counting.
// Pinned to cv2.clipLine in tests/test_line_oracle_cpu.py through the oracle's identical restatement.
__device__ __forceinline__ int line_iterator_count(int w, int h, int ax, int ay, int bx, int by) {
    long long x1 = ax, y1 = ay, x2 = bx, y2 = by;
    if ((unsigned)ax < (unsigned)w && (unsigned)bx < (unsigned)w && (unsigned)ay < (unsigned)h && (unsigned)by < (unsigned)h)
        return max(abs(bx - ax), abs(by - ay)) + 1;
    const long long right = w - 1, bottom = h - 1;
    int c1 = (x1 < 0) + (x1 > right) * 2 + (y1 < 0) * 4 + (y1 > bottom) * 8;
    int c2 = (x2 < 0) + (x2 > right) * 2 + (y2 < 0) * 4 + (y2 > bottom) * 8;
    if ((c1 & c2) == 0 && (c1 | c2) != 0) {
        long long a;
        if (c1 & 12) { a = c1 < 8 ? 0 : bottom; x1 += (a - y1) * (x2 - x1) / (y2 - y1); y1 = a; c1 = (x1 < 0) + (x1 > right) * 2; }
        if (c2 & 12) { a = c2 < 8 ? 0 : bottom; x2 += (a - y2) * (x2 - x1) / (y2 - y1); y2 = a; c2 = (x2 < 0) + (x2 > right) * 2; }
        if ((c1 & c2) == 0 && (c1 | c2) != 0) {
            if (c1) { a = c1 == 1 ? 0 : right; y1 += (a - x1) * (y2 - y1) / (x2 - x1); x1 = a; c1 = 0; }
            if (c2) { a = c2 == 1 ? 0 : right; y2 += (a - x2) * (y2 - y1) / (x2 - x1); x2 = a; c2 = 0; }
        }
    }
    if ((c1 | c2) != 0) return 0;
    const long long dx = x2 > x1 ? x2 - x1 : x1 - x2, dy = y2 > y1 ? y2 - y1 : y1 - y2;
    return (int)(dx > dy ? dx : dy) + 1;
}

// -------------------------------------------------------------------------------------------------
// KeyLine packaging (line_descriptor LSDDetector::detectImpl), top-N by response (ExtractLineSegment.cpp:45-51),
// line equations (:56-68).  One CTA per frame.
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_keylines(const __grid_constant__ LineGeom g, LineWs ws) {
    __shared__ int s_warp[33];
    const int f = blockIdx.x, tid = threadIdx.x;
    // accepted jobs -> raw segment list, in detection order
    const int nj = ws.njobs[f];
    int* flag = ws.jobflag + (long long)f * g.seg_cap;
    const int n = block_scan_array(flag, nj, s_warp);              // exclusive offsets in place
    double* segw = ws.seg + (long long)f * g.seg_cap * 4;
    const double* jobs = ws.jobs + (long long)f * g.seg_cap * 13;
    for (int j = tid; j < nj; j += 256)
        if (jobs[(long long)j * 13 + 12] > 0.0) { const int o = flag[j]; for (int k = 0; k < 4; k++) segw[4 * o + k] = jobs[(long long)j * 13 + k]; }
    if (tid == 0) { ws.nseg[f] = n; if (g.trace_cap) ws.ntrace[f] = min(nj, g.trace_cap); }
    __syncthreads();
    const double* seg = segw;
    float* resp = ws.resp + (long long)f * g.seg_cap;
    float4* ext = ws.ext + (long long)f * g.seg_cap;
    const double SCALE = 0.8;
    for (int i = tid; i < n; i += 256) {
        float e[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            double v = seg[4 * i + k] + 0.5;
            v /= SCALE;
            float fv = (float)v;
            const int lim = (k & 1) ? g.h : g.w;                       // checkLineExtremes
            if (fv < 0) fv = 0;
            if (fv >= (float)lim) fv = (float)lim - 1.0f;
            e[k] = fv;
        }
        ext[i] = make_float4(e[0], e[1], e[2], e[3]);
        const float ddx = e[0] - e[2], ddy = e[1] - e[3];
        const float len = (float)sqrt((double)ddx * (double)ddx + (double)ddy * (double)ddy);
        resp[i] = len / (float)max(g.w, g.h);
    }
    __syncthreads();
    const int keep = min(n, g.kl_cap);
    sslpl_keyline* KL = ws.kl + (long long)f * g.kl_cap;
    double* EQ = ws.lineeq + (long long)f * g.kl_cap * 3;
    for (int i = tid; i < n; i += 256) {
        int pos = i;
        if (n > g.kl_cap) {                       // stable rank by descending response
            const float r = resp[i];
            int rank = 0;
            for (int j = 0; j < n; j++) { const float rj = resp[j]; rank += (rj > r) || (rj == r && j < i); }
            pos = rank;
        }
        if (pos >= keep) continue;
        const float4 e = ext[i];
        sslpl_keyline k;
        k.startPointX = e.x; k.startPointY = e.y; k.endPointX = e.z; k.endPointY = e.w;
        k.sPointInOctaveX = e.x; k.sPointInOctaveY = e.y; k.ePointInOctaveX = e.z; k.ePointInOctaveY = e.w;
        const float ddx = e.x - e.z, ddy = e.y - e.w;
        k.lineLength = (float)sqrt((double)ddx * (double)ddx + (double)ddy * (double)ddy);
        const int ax = __float2int_rn(e.x), ay = __float2int_rn(e.y), bx = __float2int_rn(e.z), by = __float2int_rn(e.w);
        k.numOfPixels = line_iterator_count(g.w, g.h, ax, ay, bx, by);  // cv::LineIterator(8-connected).count (after cv::clipLine)
        k.angle = (float)atan2((double)(e.w - e.y), (double)(e.z - e.x));
        k.class_id = pos; k.octave = 0;
        k.size = (e.z - e.x) * (e.w - e.y);
        k.response = resp[i];
        k.pt_x = (e.z + e.x) / 2; k.pt_y = (e.w + e.y) / 2;
        KL[pos] = k;
        const double sx = e.x, sy = e.y, ex = e.z, ey = e.w;
        const double l0 = sy * 1.0 - 1.0 * ey, l1 = 1.0 * ex - sx * 1.0, l2 = sx * ey - sy * ex;
        const double nrm = sqrt(l0 * l0 + l1 * l1);
        EQ[3 * pos] = l0 / nrm; EQ[3 * pos + 1] = l1 / nrm; EQ[3 * pos + 2] = l2 / nrm;
    }
    if (tid == 0) ws.nl[f] = keep;
}

// Sobel 3x3 -> s16 (dx, dy) with BORDER_REFLECT_101 on the 5-tap blurred image.  Four pixels per thread: three
// aligned 32-bit row loads (+ the two edge bytes) and two 8-byte stores instead of 8 byte loads and 2 short stores per pixel.
__global__ void __launch_bounds__(256) k_sobel(const __grid_constant__ LineGeom g, LineWs ws) {
    const int x0 = (blockIdx.x * 32 + threadIdx.x) * 4, y = blockIdx.y * 8 + threadIdx.y, f = blockIdx.z;
    if (x0 >= g.w || y >= g.h) return;
    const uint8_t* img = ws.blur5 + f * g.blur_stride;
    const uint8_t* rows[3] = {img + (long long)reflect101(y - 1, g.h) * g.bpitch, img + (long long)y * g.bpitch, img + (long long)reflect101(y + 1, g.h) * g.bpitch};
    const int xl = reflect101(x0 - 1, g.w);
    int v[3][6];                                             // columns x0-1 .. x0+4 of the three rows
#pragma unroll
    for (int r = 0; r < 3; r++) {
        const unsigned wv = *reinterpret_cast<const unsigned*>(rows[r] + x0);     // bpitch % 64 == 0, x0 % 4 == 0; x0+3 < bpitch
        v[r][0] = rows[r][xl];
        v[r][1] = wv & 0xff; v[r][2] = (wv >> 8) & 0xff; v[r][3] = (wv >> 16) & 0xff; v[r][4] = wv >> 24;
        v[r][5] = rows[r][reflect101(min(x0 + 4, g.w), g.w)];
    }
    // pixels beyond the last column (only when w % 4 != 0) take the reflected neighbours the scalar definition uses
    short dxs[4], dys[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int x = x0 + k;
        int m0 = v[0][k], m1 = v[1][k], m2 = v[2][k], c0 = v[0][k + 1], c2 = v[2][k + 1], p0 = v[0][k + 2], p1 = v[1][k + 2], p2 = v[2][k + 2];
        if (x == g.w - 1) { p0 = m0; p1 = m1; p2 = m2; }    // reflect101(w) = w - 2 = x - 1
        dxs[k] = (short)((p0 - m0) + 2 * (p1 - m1) + (p2 - m2));
        dys[k] = (short)((m2 - m0) + 2 * (c2 - c0) + (p2 - p0));
    }
    const long long o = f * g.full_stride + (long long)y * g.w + x0;
    if ((g.w & 3) == 0 && (g.full_stride & 3) == 0) {
        *reinterpret_cast<short4*>(ws.dx + o) = make_short4(dxs[0], dxs[1], dxs[2], dxs[3]);
        *reinterpret_cast<short4*>(ws.dy + o) = make_short4(dys[0], dys[1], dys[2], dys[3]);
    } else {
#pragma unroll
        for (int k = 0; k < 4; k++) if (x0 + k < g.w) { ws.dx[o + k] = dxs[k]; ws.dy[o + k] = dys[k]; }
    }
}

// LBD (BinaryDescriptor::computeLBD, binary_descriptor.cpp) — one CTA (64 threads) per line: thread h walks row h
// of the 63-row line support region sequentially (float sums keep the reference's order), thread 0 folds the rows
// into the 9 bands in row order, then builds the 72-float vector and the 32 pair-comparison bytes.
struct LbdCoef { float G[63]; float L[21]; };
__constant__ int c_comb[32][2] = {{0, 1}, {0, 2}, {0, 3}, {0, 4}, {0, 5}, {0, 6}, {1, 2}, {1, 3}, {1, 4}, {1, 5}, {1, 6}, {2, 3}, {2, 4}, {2, 5}, {2, 6}, {2, 7},
                                  {2, 8}, {3, 4}, {3, 5}, {3, 6}, {3, 7}, {3, 8}, {4, 5}, {4, 6}, {4, 7}, {4, 8}, {5, 6}, {5, 7}, {5, 8}, {6, 7}, {6, 8}, {7, 8}};

__global__ void __launch_bounds__(64) k_lbd(const __grid_constant__ LineGeom g, LineWs ws, const __grid_constant__ LbdCoef C) {
    __shared__ float s_row[63][8];
    __shared__ float s_des[72];
    const int li = blockIdx.x, f = blockIdx.y, h = threadIdx.x;
    if (li >= ws.nl[f]) return;
    const sslpl_keyline kl = ws.kl[(long long)f * g.kl_cap + li];
    const int16_t* dxI = ws.dx + f * g.full_stride; const int16_t* dyI = ws.dy + f * g.full_stride;
    const short imageWidth = (short)(g.w - 1), imageHeight = (short)(g.h - 1);
    const short lengthOfLSP = (short)kl.numOfPixels, halfWidth = (short)((lengthOfLSP - 1) / 2), halfHeight = 31;
    const float mx = (float)(0.5 * (double)(kl.sPointInOctaveX + kl.ePointInOctaveX));
    const float my = (float)(0.5 * (double)(kl.sPointInOctaveY + kl.ePointInOctaveY));
    const float dL0 = (float)cos((double)kl.angle), dL1 = (float)sin((double)kl.angle);
    const float dO0 = -dL1, dO1 = dL0;
    if (h < 63) {
        // sCorX0 after h steps of (sCorX0 -= dL[1]; sCorY0 += dL[0]) — replay the float recurrence exactly
        float sx0 = -dL0 * halfWidth + dL1 * halfHeight + mx;
        float sy0 = -dL1 * halfWidth - dL0 * halfHeight + my;
        for (int k = 0; k < h; k++) { sx0 -= dL1; sy0 += dL0; }
        float sx = sx0, sy = sy0, pL = 0, nL = 0, pO = 0, nO = 0;
        for (short wID = 0; wID < lengthOfLSP; wID++) {
            short t = (short)roundf(sx);
            const short xc = (t < 0) ? 0 : (t > imageWidth) ? imageWidth : t;
            t = (short)roundf(sy);
            const short yc = (t < 0) ? 0 : (t > imageHeight) ? imageHeight : t;
            const short dx = dxI[(int)yc * g.w + xc], dy = dyI[(int)yc * g.w + xc];
            const float gDL = dx * dL0 + dy * dL1, gDO = dx * dO0 + dy * dO1;
            if (gDL > 0) pL += gDL; else nL -= gDL;
            if (gDO > 0) pO += gDO; else nO -= gDO;
            sx += dL0; sy += dL1;
        }
        const float cg = C.G[h];
        pL = cg * pL; nL = cg * nL; pO = cg * pO; nO = cg * nO;
        s_row[h][0] = pL; s_row[h][1] = nL; s_row[h][2] = pL * pL; s_row[h][3] = nL * nL;
        s_row[h][4] = pO; s_row[h][5] = nO; s_row[h][6] = pO * pO; s_row[h][7] = nO * nO;
    }
    __syncthreads();
    if (h < 8) {      // thread q accumulates quantity q of every band, rows in order (same add order as the reference)
        float band[9];
#pragma unroll
        for (int b = 0; b < 9; b++) band[b] = 0;
        const bool sq = (h & 2) != 0;           // quantities 2,3,6,7 use squared local weights
        for (int r = 0; r < 63; r++) {
            const float v = s_row[r][h];
            int b = r / 7;
            float c = C.L[r % 7 + 7];
            band[b] += (sq ? c * c : c) * v;
            b--;
            if (b >= 0) { c = C.L[r % 7 + 14]; band[b] += (sq ? c * c : c) * v; }
            b += 2;
            if (b < 9) { c = C.L[r % 7]; band[b] += (sq ? c * c : c) * v; }
        }
        for (int b = 0; b < 9; b++) s_row[b][h] = band[b];      // reuse rows 0..8 as band sums (all reads are done: see sync)
    }
    __syncthreads();
    if (h == 0) {
        const float invN2 = (float)(1.0 / (7 * 2.0)), invN3 = (float)(1.0 / (7 * 3.0));
        float* d = s_des;
        for (int b = 0; b < 9; b++) {
            const float invN = (b == 0 || b == 8) ? invN2 : invN3;
            float t = s_row[b][0] * invN; d[8 * b] = t; d[8 * b + 4] = sqrtf(s_row[b][2] * invN - t * t);
            t = s_row[b][1] * invN; d[8 * b + 1] = t; d[8 * b + 5] = sqrtf(s_row[b][3] * invN - t * t);
            t = s_row[b][4] * invN; d[8 * b + 2] = t; d[8 * b + 6] = sqrtf(s_row[b][6] * invN - t * t);
            t = s_row[b][5] * invN; d[8 * b + 3] = t; d[8 * b + 7] = sqrtf(s_row[b][7] * invN - t * t);
        }
        float tM = 0, tS = 0;
        for (int b = 0; b < 9; b++) {
            for (int i = 0; i < 4; i++) tM += d[8 * b + i] * d[8 * b + i];
            for (int i = 4; i < 8; i++) tS += d[8 * b + i] * d[8 * b + i];
        }
        tM = 1 / sqrtf(tM); tS = 1 / sqrtf(tS);
        for (int b = 0; b < 9; b++) {
            for (int i = 0; i < 4; i++) d[8 * b + i] = d[8 * b + i] * tM;
            for (int i = 4; i < 8; i++) d[8 * b + i] = d[8 * b + i] * tS;
        }
        for (int i = 0; i < 72; i++) if ((double)d[i] > 0.4) d[i] = (float)0.4;
        float t = 0;
        for (int i = 0; i < 72; i++) t += d[i] * d[i];
        t = 1 / sqrtf(t);
        for (int i = 0; i < 72; i++) d[i] = d[i] * t;
    }
    __syncthreads();
    if (h < 32) {
        const float* f1 = &s_des[8 * c_comb[h][0]]; const float* f2 = &s_des[8 * c_comb[h][1]];
        unsigned r = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) if (f1[i] > f2[i]) r += 0x80u >> i;
        // 32 bytes -> two coalesced 16-byte stores
        uint32_t w = r << (8 * (h & 3));
        w |= __shfl_xor_sync(0xffffffffu, w, 1);
        w |= __shfl_xor_sync(0xffffffffu, w, 2);
        const uint32_t w0 = __shfl_sync(0xffffffffu, w, (h & 16) + 0), w1 = __shfl_sync(0xffffffffu, w, (h & 16) + 4),
                       w2 = __shfl_sync(0xffffffffu, w, (h & 16) + 8), w3 = __shfl_sync(0xffffffffu, w, (h & 16) + 12);
        if ((h & 15) == 0) reinterpret_cast<uint4*>(ws.ldesc + ((long long)f * g.kl_cap + li) * 32)[h >> 4] = make_uint4(w0, w1, w2, w3);
    }
}

}  // namespace sslpl

// =================================================================================================
using namespace sslpl;

struct sslpl_line {
    sslpl_line_params p;
    cudaStream_t stream = nullptr, own_stream = nullptr;
    uint8_t* arena = nullptr; size_t arena_size = 0;
    LineGeom g; LineWs ws; LView view;
    uint8_t* d_input = nullptr;
    LbdCoef coef;
    bool trace = false;
    int used_smem = 0;
    int sm_count = 148;
    int max_walkers = 0;        // 0 = one walker CTA per frame
    int walker_warps = 0;       // 0 = automatic (one warp or 16 warps per frame), -1 = one warp
    int cur_w = 0, cur_h = 0, cur_frames = 0;
    long long launches = 0;
    int* h_err = nullptr;
    bool profiling = false;
    std::vector<cudaEvent_t> ev; std::vector<const char*> ev_name; int ev_n = 0;
};

namespace {

void lmark(sslpl_line* h, const char* name) {
    if (!h->profiling) return;
    if ((int)h->ev.size() <= h->ev_n) { cudaEvent_t e; cudaEventCreate(&e); h->ev.push_back(e); h->ev_name.push_back(name); }
    h->ev_name[h->ev_n] = name;
    cudaEventRecord(h->ev[h->ev_n++], h->stream);
}

void make_geometry(const sslpl_line* h, int W, int H, LineGeom& g, std::vector<int2>* tab) {
    memset(&g, 0, sizeof(g));
    g.w = W; g.h = H; g.pitch = (int)align_up(W, 16);
    g.bpitch = (int)align_up(W, 64);
    g.sw = (int)lrint(W * 0.8); g.sh = (int)lrint(H * 0.8); g.spitch = (int)align_up(g.sw, 64);
    g.tiles_x = (W + LT_W - 1) / LT_W; g.tiles_y = (H + LT_H - 1) / LT_H;
    g.xtab_off = 0; g.ytab_off = g.sw;
    g.in_stride = (long long)g.pitch * H;
    g.blur_stride = (long long)align_up((size_t)g.bpitch * H, 256);
    g.scaled_stride = (long long)align_up((size_t)g.spitch * g.sh, 256);
    g.pix_stride = (long long)g.sw * g.sh;
    g.full_stride = (long long)W * H;
    g.kl_cap = h->p.lsdNFeatures;
    // lsd.cpp constants (ANG_TH 22.5, QUANT 2.0); host libm, exactly as the CPU implementation evaluates them
    g.prec = L_PI * 22.5 / 180; g.p = 22.5 / 180; g.rho = 2.0 / std::sin(g.prec);
    g.log_nt = 5 * (std::log10(double(g.sw)) + std::log10(double(g.sh))) / 2 + std::log10(11.0);
    g.min_reg_size = (int)size_t(-g.log_nt / std::log10(g.p));
    g.seg_cap = (int)(g.pix_stride / std::max(g.min_reg_size, 1)) + 16;
    g.trace_cap = h->trace ? g.seg_cap : 0;
    g.dbg = getenv("SSLPL_WALKER_DBG") ? atoi(getenv("SSLPL_WALKER_DBG")) : 0;
    if (tab) {
        tab->assign(g.sw + g.sh, make_int2(0, 0));
        for (int axis = 0; axis < 2; axis++) {
            const int dn = axis ? g.sh : g.sw, sn = axis ? H : W, off = axis ? g.ytab_off : g.xtab_off;
            // cv::resize(..., Size(), 0.8, 0.8, INTER_LINEAR_EXACT) maps with scale = 1 / fx = 1.25, not sn / dn (resize.cpp)
            const double sc = 1.0 / 0.8; (void)sn;
            for (int d = 0; d < dn; d++) {
                double s = (d + 0.5) * sc - 0.5;
                int i0 = (int)floor(s);
                double f = s - i0;
                if (i0 < 0) { i0 = 0; f = 0; }
                if (i0 >= sn - 1) { i0 = sn - 1; f = 0; }
                (*tab)[off + d] = make_int2(i0, (int)lrint(f * 256));
            }
        }
    }
}

void carve(sslpl_line* h, Arena& A, const LineGeom& g, int B) {
    LineWs& ws = h->ws;
    h->d_input = A.take<uint8_t>((size_t)B * g.in_stride + 256);
    ws.blur7 = A.take<uint8_t>((size_t)B * g.blur_stride); ws.blur5 = A.take<uint8_t>((size_t)B * g.blur_stride);
    ws.scaled = A.take<uint8_t>((size_t)B * g.scaled_stride);
    ws.angdeg = A.take<float>((size_t)B * g.pix_stride); ws.pix = A.take<LPix>((size_t)B * g.pix_stride);
    ws.modgrad = A.take<double>((size_t)B * g.pix_stride); ws.cs0 = A.take<float2>((size_t)B * g.pix_stride);
    ws.maxgrad = A.take<unsigned long long>(B);
    ws.seeds = A.take<unsigned>((size_t)B * g.pix_stride); ws.nseeds = A.take<int>(B);
    ws.reg = A.take<unsigned>((size_t)B * g.pix_stride);
    ws.sreg = A.take<unsigned>((size_t)B * WALK_RING * WALK_SLOT_CAP);
    ws.wstat = A.take<unsigned long long>(16);
    ws.seg = A.take<double>((size_t)B * g.seg_cap * 4); ws.nseg = A.take<int>(B);
    ws.jobs = A.take<double>((size_t)B * g.seg_cap * 13); ws.njobs = A.take<int>(B); ws.jobflag = A.take<int>((size_t)B * g.seg_cap);
    ws.jobnk = A.take<int2>((size_t)B * g.seg_cap); ws.jobnfa = A.take<double>((size_t)B * g.seg_cap);
    ws.rej = A.take<int2>((size_t)B * g.seg_cap); ws.rejctl = A.take<int>(4);

    ws.dx = A.take<int16_t>((size_t)B * g.full_stride); ws.dy = A.take<int16_t>((size_t)B * g.full_stride);
    ws.tab = A.take<int2>(g.sw + g.sh);
    ws.resp = A.take<float>((size_t)B * g.seg_cap); ws.ext = A.take<float4>((size_t)B * g.seg_cap);
    ws.kl = A.take<sslpl_keyline>((size_t)B * g.kl_cap); ws.ldesc = A.take<uint8_t>((size_t)B * g.kl_cap * 32);
    ws.lineeq = A.take<double>((size_t)B * g.kl_cap * 3); ws.nl = A.take<int>(B);
    ws.err = A.take<int>(1);
    ws.trace = A.take<double>((size_t)B * g.trace_cap * 10 + 16); ws.ntrace = A.take<int>(B);
    ws.lgam = A.take<double>((size_t)g.pix_stride + 2);
}

// log_gamma of lsd.cpp on the host (same libm as the CPU implementation): Lanczos for x <= 15, Windschitl above
double host_log_gamma(double x) {
    if (x > 15.0) return 0.918938533204673 + (x - 0.5) * std::log(x) - x + 0.5 * x * std::log(x * std::sinh(1 / x) + 1 / (810.0 * std::pow(x, 6.0)));
    static const double q[7] = {75122.6331530, 80916.6278952, 36308.2951477, 8687.24529705, 1168.92649479, 83.8676043424, 2.50662827511};
    double a = (x + 0.5) * std::log(x + 5.5) - (x + 5.5), b = 0;
    for (int n = 0; n < 7; ++n) { a -= std::log(x + double(n)); b += q[n] * std::pow(x, double(n)); }
    return a + std::log(b);
}

int configure(sslpl_line* h, int W, int H) {
    if (W == h->cur_w && H == h->cur_h) return SSLPL_OK;
    SSLPL_REQUIRE(W <= h->p.max_width && H <= h->p.max_height, SSLPL_ERR_ARG, "frame larger than the handle's max_width/max_height");
    SSLPL_REQUIRE(W >= 16 && H >= 16 && W < 32768 && H < 32768, SSLPL_ERR_ARG, "frame size out of range");
    std::vector<int2> tab;
    make_geometry(h, W, H, h->g, &tab);
    Arena A; A.base = h->arena; A.size = h->arena_size;
    carve(h, A, h->g, h->p.max_batch);
    SSLPL_REQUIRE(A.used <= h->arena_size, SSLPL_ERR_CAPACITY, "internal: arena too small for this frame size");
    SSLPL_CUDA(cudaStreamSynchronize(h->stream));
    SSLPL_CUDA(cudaMemcpy(h->ws.tab, tab.data(), tab.size() * sizeof(int2), cudaMemcpyHostToDevice));
    SSLPL_CUDA(cudaMemset(h->ws.err, 0, sizeof(int)));
    {
        std::vector<double> lg((size_t)h->g.pix_stride + 2);
        for (size_t n = 0; n < lg.size(); n++) lg[n] = host_log_gamma((double)n + 1.0);
        SSLPL_CUDA(cudaMemcpy(const_cast<double*>(h->ws.lgam), lg.data(), lg.size() * sizeof(double), cudaMemcpyHostToDevice));
    }
    h->cur_w = W; h->cur_h = H;
    return SSLPL_OK;
}

int run_pipeline(sslpl_line* h, int B) {
    const LineGeom& g = h->g;
    cudaStream_t st = h->stream;
    const Taps7 t7 = {{0, 4, 56, 136, 56, 4, 0}};       // GaussianBlur(sigma 0.6/0.8) of lsd.cpp, 4.13 fixed point
    const Taps7 t5 = {{0, 14, 62, 104, 62, 14, 0}};     // GaussianBlur(5x5, sigma 1) of BinaryDescriptor
    const dim3 tiles(g.tiles_x * g.tiles_y, B);
    h->ev_n = 0;
    lmark(h, "start");
    k_sep7<<<tiles, 256, 0, st>>>(g, h->view, h->ws.blur7, h->ws.blur5, g.blur_stride, t7, t5);      // both blurs from one staged tile
    k_resize_exact<<<dim3((g.sw + 31) / 32, (g.sh + 7) / 8, B), dim3(32, 8), 0, st>>>(g, h->ws);
    lmark(h, "lsd_prep");
    SSLPL_CUDA(cudaMemsetAsync(h->ws.maxgrad, 0, sizeof(unsigned long long) * B, st));
    k_ll_angle<<<dim3((g.sw + 127) / 128, (g.sh + 7) / 8, B), dim3(32, 8), 0, st>>>(g, h->ws);
    lmark(h, "lsd_ll_angle");
    k_lsd_seeds<<<B, SEED_WARPS * 32, 0, st>>>(g, h->ws);
    lmark(h, "lsd_seeds");
    SSLPL_CUDA(cudaMemsetAsync(h->ws.rejctl, 0, 4 * sizeof(int), st));
    SSLPL_CUDA(cudaMemsetAsync(h->ws.wstat, 0, 16 * sizeof(unsigned long long), st));
    {   // one CTA per frame; few frames -> more warps per frame (latency), many frames -> more CTAs per SM (throughput)
        // automatic choice (measured, B200): big batches (at least two frames per SM) -> one warp per frame (k_lsd_regions_solo);
        // fewer frames -> the multi-warp walker k_lsd_regions with 16 warps per frame.  SSLPL_WALKER_WARPS overrides it (-1 = one warp).
        const int ww = h->walker_warps < 0 ? 0 : h->walker_warps > 0 ? std::min(h->walker_warps, WALK_MAXW) : (B >= 2 * h->sm_count ? 0 : WALK_MAXW);
        const size_t smem = (size_t)((g.pix_stride + 31) / 32) * sizeof(unsigned);
        if ((int)smem > h->used_smem) { SSLPL_CUDA(cudaFuncSetAttribute(k_lsd_regions, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); h->used_smem = (int)smem; }
        const int grid = h->max_walkers > 0 ? std::min(B, h->max_walkers) : B;
        if (ww == 0) k_lsd_regions_solo<<<grid, 32, 0, st>>>(g, h->ws, B);
        else k_lsd_regions<<<grid, ww * 32, smem, st>>>(g, h->ws, B);
    }
    lmark(h, "lsd_regions");
    k_lsd_nfa_count<<<dim3(NFA_COUNT_CTAS, B), 128, 0, st>>>(g, h->ws);
    k_lsd_nfa_first<<<dim3(NFA_FIRST_CTAS, B), 128, 0, st>>>(g, h->ws);
    k_lsd_nfa_improve<<<std::min(h->sm_count * 8, (B * 64 + 3) / 4), 128, 0, st>>>(g, h->ws);
    lmark(h, "lsd_nfa");
    k_keylines<<<B, 256, 0, st>>>(g, h->ws);
    k_sobel<<<dim3((g.w + 127) / 128, (g.h + 7) / 8, B), dim3(32, 8), 0, st>>>(g, h->ws);
    k_lbd<<<dim3(g.kl_cap, B), 64, 0, st>>>(g, h->ws, h->coef);
    lmark(h, "keylines_lbd");
    h->launches += 11;     // kernels only (the two small memsets are not counted)
    SSLPL_CUDA(cudaGetLastError());
    return SSLPL_OK;
}

int check_device_err(sslpl_line* h) {
    if (h->cur_w == 0) { SSLPL_CUDA(cudaStreamSynchronize(h->stream)); return SSLPL_OK; }     // never used yet: no workspace, nothing to report
    SSLPL_CUDA(cudaMemcpyAsync(h->h_err, h->ws.err, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    SSLPL_CUDA(cudaStreamSynchronize(h->stream));
    if (*h->h_err) {
        set_error("device-side capacity overflow in the line path, flags=0x%x", *h->h_err);
        cudaMemsetAsync(h->ws.err, 0, sizeof(int), h->stream);
        return SSLPL_ERR_CAPACITY;
    }
    return SSLPL_OK;
}

}  // namespace

extern "C" {

int sslpl_line_create(const sslpl_line_params* p, sslpl_line** out) {
    SSLPL_REQUIRE(p && out, SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(p->lsdNFeatures >= 1 && p->lsdNFeatures <= 65536, SSLPL_ERR_ARG, "lsdNFeatures out of range");
    SSLPL_REQUIRE(p->max_batch >= 1 && p->max_width >= 16 && p->max_height >= 16, SSLPL_ERR_ARG, "bad max_batch / max size");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) { set_error("no CUDA device available: libsslpl_b200 has no CPU fallback"); return SSLPL_ERR_CUDA; }
    SSLPL_CUDA(cudaSetDevice(p->device));
    sslpl_line* h = new sslpl_line();
    h->p = *p;
    { int v = 0; if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, p->device) == cudaSuccess && v > 0) h->sm_count = v; }
    h->trace = getenv("SSLPL_LINE_TRACE") != nullptr;
    if (const char* e = getenv("SSLPL_WALKER_WARPS")) h->walker_warps = std::max(-1, std::min(WALK_MAXW, atoi(e)));   // tuning knob (tests sweep it); -1 = the one-warp throughput kernel
    {   // BinaryDescriptor constructor: local (F_l) and global (F_g) Gaussian weights, widthOfBand 7, 9 bands
        double u = (7 * 3 - 1) / 2, sigma = (7 * 2 + 1) / 2, inv = -1 / (2 * sigma * sigma);
        for (int i = 0; i < 21; i++) { const double d = i - u; h->coef.L[i] = (float)exp(d * d * inv); }
        u = (9 * 7 - 1) / 2; sigma = u; inv = -1 / (2 * sigma * sigma);
        for (int i = 0; i < 63; i++) { const double d = i - u; h->coef.G[i] = (float)exp(d * d * inv); }
    }
    LineGeom g;
    make_geometry(h, p->max_width, p->max_height, g, nullptr);
    Arena A; carve(h, A, g, p->max_batch);
    h->arena_size = A.used + (1 << 20);
    cudaError_t e = cudaMalloc(&h->arena, h->arena_size);
    if (e != cudaSuccess) { set_error("cudaMalloc(%zu) failed: %s", h->arena_size, cudaGetErrorString(e)); delete h; return SSLPL_ERR_CUDA; }
    SSLPL_CUDA(cudaMemset(h->arena, 0, h->arena_size));
    SSLPL_CUDA(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    h->stream = h->own_stream;
    SSLPL_CUDA(cudaHostAlloc((void**)&h->h_err, sizeof(int), cudaHostAllocDefault));
    *out = h;
    return SSLPL_OK;
}

void sslpl_line_destroy(sslpl_line* h) {
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

int sslpl_line_sync(sslpl_line* h) { SSLPL_REQUIRE(h, SSLPL_ERR_ARG, "null handle"); SSLPL_CUDA(cudaSetDevice(h->p.device)); return check_device_err(h); }
void* sslpl_line_stream(sslpl_line* h) { return h ? (void*)h->stream : nullptr; }
int sslpl_line_set_stream(sslpl_line* h, void* s) {
    SSLPL_REQUIRE(h, SSLPL_ERR_ARG, "null handle");
    SSLPL_CUDA(cudaSetDevice(h->p.device));
    SSLPL_CUDA(cudaStreamSynchronize(h->stream));
    h->stream = s ? (cudaStream_t)s : h->own_stream;
    return SSLPL_OK;
}
long long sslpl_line_launch_count(const sslpl_line* h) { return h ? h->launches : 0; }
int sslpl_line_set_max_walkers(sslpl_line* h, int max_concurrent) {
    SSLPL_REQUIRE(h && max_concurrent >= 0, SSLPL_ERR_ARG, "bad argument");
    h->max_walkers = max_concurrent;
    return SSLPL_OK;
}
int sslpl_line_set_profiling(sslpl_line* h, int on) { SSLPL_REQUIRE(h, SSLPL_ERR_ARG, "null handle"); h->profiling = on != 0; return SSLPL_OK; }
int sslpl_line_stage_ms(sslpl_line* h, float* ms, int cap, const char** names, int* nstages) {
    SSLPL_REQUIRE(h && nstages, SSLPL_ERR_ARG, "null argument");
    SSLPL_CUDA(cudaStreamSynchronize(h->stream));
    int k = 0;
    for (int i = 1; i < h->ev_n; i++, k++)
        if (k < cap) { float t = 0; cudaEventElapsedTime(&t, h->ev[i - 1], h->ev[i]); if (ms) ms[k] = t; if (names) names[k] = h->ev_name[i]; }
    *nstages = k;
    return SSLPL_OK;
}

int sslpl_line_extract_batch_device(sslpl_line* h, const uint8_t* d_imgs, int nframes, int width, int height, int pitch, size_t frame_stride) {
    SSLPL_REQUIRE(h && d_imgs, SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(nframes >= 1 && nframes <= h->p.max_batch && pitch >= width, SSLPL_ERR_ARG, "bad nframes / pitch");
    SSLPL_CUDA(cudaSetDevice(h->p.device));
    int rc = configure(h, width, height);
    if (rc) return rc;
    h->view.base = d_imgs; h->view.pitch = pitch; h->view.frame_stride = (long long)frame_stride;
    h->cur_frames = nframes;
    return run_pipeline(h, nframes);
}

int sslpl_line_device_results(sslpl_line* h, const sslpl_keyline** d_kl, const uint8_t** d_ldesc, const double** d_lineeq, const int** d_n, int* cap) {
    SSLPL_REQUIRE(h, SSLPL_ERR_ARG, "null handle");
    if (d_kl) *d_kl = h->ws.kl;
    if (d_ldesc) *d_ldesc = h->ws.ldesc;
    if (d_lineeq) *d_lineeq = h->ws.lineeq;
    if (d_n) *d_n = h->ws.nl;
    if (cap) *cap = h->p.lsdNFeatures;
    return SSLPL_OK;
}

int sslpl_line_extract_batch_begin(sslpl_line* h, const uint8_t* imgs, int nframes, int width, int height, int pitch, size_t frame_stride,
                                   sslpl_keyline* kl, uint8_t* ldesc, double* lineeq, int cap, int* n) {
    SSLPL_REQUIRE(h && kl && ldesc && lineeq && n && imgs, SSLPL_ERR_ARG, "null argument");
    SSLPL_REQUIRE(nframes >= 1 && nframes <= h->p.max_batch && pitch >= width, SSLPL_ERR_ARG, "bad nframes / pitch");
    SSLPL_REQUIRE(cap >= h->p.lsdNFeatures, SSLPL_ERR_CAPACITY, "caller line capacity smaller than lsdNFeatures");
    SSLPL_CUDA(cudaSetDevice(h->p.device));
    int rc = configure(h, width, height);
    if (rc) return rc;
    const LineGeom& g = h->g;
    if (frame_stride == (size_t)pitch * height)
        SSLPL_CUDA(cudaMemcpy2DAsync(h->d_input, g.pitch, imgs, pitch, width, (size_t)height * nframes, cudaMemcpyHostToDevice, h->stream));
    else
        for (int f = 0; f < nframes; f++)
            SSLPL_CUDA(cudaMemcpy2DAsync(h->d_input + f * g.in_stride, g.pitch, imgs + f * frame_stride, pitch, width, height, cudaMemcpyHostToDevice, h->stream));
    h->view.base = h->d_input; h->view.pitch = g.pitch; h->view.frame_stride = g.in_stride;
    h->cur_frames = nframes;
    rc = run_pipeline(h, nframes);
    if (rc) return rc;
    const int kc = g.kl_cap;
    SSLPL_CUDA(cudaMemcpyAsync(n, h->ws.nl, sizeof(int) * nframes, cudaMemcpyDeviceToHost, h->stream));
    SSLPL_CUDA(cudaMemcpy2DAsync(kl, (size_t)cap * sizeof(sslpl_keyline), h->ws.kl, (size_t)kc * sizeof(sslpl_keyline), (size_t)kc * sizeof(sslpl_keyline), nframes, cudaMemcpyDeviceToHost, h->stream));
    SSLPL_CUDA(cudaMemcpy2DAsync(ldesc, (size_t)cap * 32, h->ws.ldesc, (size_t)kc * 32, (size_t)kc * 32, nframes, cudaMemcpyDeviceToHost, h->stream));
    SSLPL_CUDA(cudaMemcpy2DAsync(lineeq, (size_t)cap * 24, h->ws.lineeq, (size_t)kc * 24, (size_t)kc * 24, nframes, cudaMemcpyDeviceToHost, h->stream));
    return SSLPL_OK;
}

int sslpl_line_extract_batch(sslpl_line* h, const uint8_t* imgs, int nframes, int width, int height, int pitch, size_t frame_stride,
                             sslpl_keyline* kl, uint8_t* ldesc, double* lineeq, int cap, int* n) {
    int rc = sslpl_line_extract_batch_begin(h, imgs, nframes, width, height, pitch, frame_stride, kl, ldesc, lineeq, cap, n);
    if (rc) return rc;
    return check_device_err(h);
}

int sslpl_line_extract(sslpl_line* h, const uint8_t* img, int width, int height, int pitch, sslpl_keyline* kl, uint8_t* ldesc, double* lineeq, int cap, int* n) {
    return sslpl_line_extract_batch(h, img, 1, width, height, pitch, (size_t)pitch * height, kl, ldesc, lineeq, cap, n);
}

int sslpl_line_download_segments(sslpl_line* h, int frame, float* seg4, int cap, int* n) {
    SSLPL_REQUIRE(h && n && frame >= 0 && frame < h->cur_frames, SSLPL_ERR_ARG, "bad argument");
    SSLPL_CUDA(cudaSetDevice(h->p.device));
    SSLPL_CUDA(cudaStreamSynchronize(h->stream));
    int cnt = 0;
    SSLPL_CUDA(cudaMemcpy(&cnt, h->ws.nseg + frame, sizeof(int), cudaMemcpyDeviceToHost));
    std::vector<double> s((size_t)std::max(cnt, 1) * 4);
    if (cnt) SSLPL_CUDA(cudaMemcpy(s.data(), h->ws.seg + (size_t)frame * h->g.seg_cap * 4, sizeof(double) * 4 * cnt, cudaMemcpyDeviceToHost));
    for (int i = 0; i < cnt && i < cap; i++)
        for (int k = 0; k < 4; k++) { double v = s[4 * i + k] + 0.5; v /= 0.8; seg4[4 * i + k] = (float)v; }
    *n = cnt;
    return SSLPL_OK;
}


/* debug (SSLPL_LINE_TRACE=1 at handle creation): one row of 10 doubles per region that reached region2rect */
/* Statistics of the last region-walker launch (16 values; collected with SSLPL_WALKER_DBG=32 by the multi-warp walker k_lsd_regions):
   [0] regions grown by the turn holder, [1] their clock cycles, [2] their pixels, [3] -, [4] claims whose seed had been swallowed
   by commit time, [5] redone by the turn holder: abandoned, [6] poisoned, [7] failed validation, [8] presumed swallowed but not,
   [9] attempts committed as speculated, [10] their pixels, [11] cycles under the commit lock, [12] under the claim lock, [13] attempts
   repeated after a lower rank retired, [14] cycles per frame (summed), [15] claims. */
int sslpl_line_walker_stats(sslpl_line* h, unsigned long long* out16) {
    SSLPL_REQUIRE(h && out16, SSLPL_ERR_ARG, "null argument");
    SSLPL_CUDA(cudaSetDevice(h->p.device));
    SSLPL_CUDA(cudaStreamSynchronize(h->stream));
    SSLPL_CUDA(cudaMemcpy(out16, h->ws.wstat, 16 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return SSLPL_OK;
}
int sslpl_line_debug_trace(sslpl_line* h, int frame, double* out, int cap_rows, int* n) {
    SSLPL_REQUIRE(h && n && frame >= 0 && frame < h->cur_frames, SSLPL_ERR_ARG, "bad argument");
    SSLPL_REQUIRE(h->g.trace_cap > 0, SSLPL_ERR_UNSUPPORTED, "tracing is off (set SSLPL_LINE_TRACE=1 before creating the handle)");
    SSLPL_CUDA(cudaSetDevice(h->p.device));
    SSLPL_CUDA(cudaStreamSynchronize(h->stream));
    int cnt = 0;
    SSLPL_CUDA(cudaMemcpy(&cnt, h->ws.ntrace + frame, sizeof(int), cudaMemcpyDeviceToHost));
    const int m = std::min(cnt, cap_rows);
    if (m > 0) SSLPL_CUDA(cudaMemcpy(out, h->ws.trace + (size_t)frame * h->g.trace_cap * 10, sizeof(double) * 10 * m, cudaMemcpyDeviceToHost));
    *n = cnt;
    return SSLPL_OK;
}

}  // extern "C"
