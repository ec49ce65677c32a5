// roi_align.cu -- K5: FPN level-mapped RoIAlign forward (BasicRoIExtractor,
// lib/region.py:243-306, on torchvision RoIAlign semantics, aligned=False by
// default) for all images and levels in ONE launch, output rows in the original
// RoI order (replaces the per-level boolean gather/scatter of lib/region.py:290-295).
//
// Arithmetic follows torchvision's CPU kernel operation by operation (bilinear
// weights hy*hx.., ((w1*v1 + w2*v2) + w3*v3) + w4*v4, sample sum, one divide by
// the sample count) with FMA contraction disabled, so results are bit-identical to
// the reference on CPU, far inside the 1e-5 north_star tolerance.
//
//   k_roi_align_win   NHWC, 2x2 samples per bin (every reference config): one CTA per (RoI,
//                     128-channel tile), lanes across channels; the distinct tap cells of a
//                     bin are loaded once as coalesced 128-bit channel quads, all loads of a
//                     bin in flight together; the [C,7,7] result is staged in shared memory
//                     in its HBM layout and leaves as one bulk async store.
//   k_roi_align_nhwc  NHWC, any fixed sampling ratio: per-sample tap descriptors in smem.
//   k_roi_align_any   generic fallback (NCHW input, adaptive sampling, odd shapes):
//                     one thread per output element, pw fastest.
// HBM roofline: 50 176 B/RoI of output + the touched feature cells (SURVEY 8(d)).
#include <cuda_bf16.h>

#include <cstdlib>
#include <cstring>

#include "roi_common.cuh"

namespace b2d {

__global__ void __launch_bounds__(256) k_roi_levels(int* __restrict__ levels, const float* __restrict__ rois,
                                                    long long ld, long long R, float finest, int num_levels) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    levels[r] = roi_level(rois[r], rois[ld + r], rois[2 * ld + r], rois[3 * ld + r], finest, num_levels);
}

constexpr int kCTile = 256;      // channels per shared-memory tile

__device__ __forceinline__ float4 ld4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float4 ld4(const __nv_bfloat16* p) {
    const uint2 u = __ldg(reinterpret_cast<const uint2*>(p));
    const __nv_bfloat162 a = *reinterpret_cast<const __nv_bfloat162*>(&u.x);
    const __nv_bfloat162 b = *reinterpret_cast<const __nv_bfloat162*>(&u.y);
    const float2 fa = __bfloat1622float2(a), fb = __bfloat1622float2(b);
    return make_float4(fa.x, fa.y, fb.x, fb.y);
}

// Per-sample descriptor staged in shared memory: element offsets of the 4 taps (relative
// to the image's feature base, channel 0) and their bilinear weights.  Invalid samples
// (outside (-1, size)) get zero weights, exactly like torchvision's pre-calc table.
struct __align__(16) Tap4 { int o1, o2, o3, o4; float w1, w2, w3, w4; };

constexpr int kMaxSamples = 256;   // PH*PW*sr*sr limit of the fast kernel (7*7*2*2 = 196)

template <typename FT>
__global__ void __launch_bounds__(256) k_roi_align_nhwc(RoiArgs a, float* __restrict__ out) {
    extern __shared__ __align__(16) float s_tile[];                      // [bins][kCTile + 4]
    __shared__ Tap4 s_tap[kMaxSamples];
    const long long r = blockIdx.x;
    const b2d_roi_cfg& c = a.cfg;
    float x1, y1, x2, y2;
    int img;
    if (!roi_fetch(a, r, img, x1, y1, x2, y2)) return;
    int lvl;
    if (a.levels) lvl = a.levels[r];
    else lvl = c.num_levels > 1 ? roi_level(x1, y1, x2, y2, c.finest_scale, c.num_levels) : 0;
    const int H = c.H[lvl], W = c.W[lvl], C = c.C;
    const RoiGeom g = roi_geom(x1, y1, x2, y2, c.spatial_scale[lvl], c.PH, c.PW, c.sampling_ratio, c.aligned);
    const int spb = g.gy * g.gx;                           // samples per bin
    const int bins = c.PH * c.PW;
    {   // sample t = ((ph*PW + pw)*gy + iy)*gx + ix  (torchvision's pre-calc order)
        const int t = threadIdx.x;
        if (t < bins * spb) {
            const int ix = t % g.gx, iy = (t / g.gx) % g.gy;
            const int bin = t / spb, ph = bin / c.PW, pw = bin - ph * c.PW;
            const AxisTap ty = axis_tap(g.sy, g.bh, ph, iy, g.gy, H);
            const AxisTap tx = axis_tap(g.sx, g.bw, pw, ix, g.gx, W);
            Tap4 q;
            if (ty.valid && tx.valid) {
                q.o1 = (ty.lo * W + tx.lo) * C; q.o2 = (ty.lo * W + tx.hi) * C;
                q.o3 = (ty.hi * W + tx.lo) * C; q.o4 = (ty.hi * W + tx.hi) * C;
                q.w1 = ty.h * tx.h; q.w2 = ty.h * tx.l; q.w3 = ty.l * tx.h; q.w4 = ty.l * tx.l;
            } else {
                q.o1 = q.o2 = q.o3 = q.o4 = 0; q.w1 = q.w2 = q.w3 = q.w4 = 0.0f;
            }
            s_tap[t] = q;
        }
    }
    __syncthreads();
    const FT* feat = reinterpret_cast<const FT*>(a.feat[lvl]) + (long long)img * H * W * C;
    const int pitch = kCTile + 4;
    const float cnt = (float)max(spb, 1);
    const int cq = threadIdx.x & 63, grp = threadIdx.x >> 6;
    float* o = out + r * (long long)C * bins;
    for (int c0 = 0; c0 < C; c0 += kCTile) {
        const int ch = c0 + cq * 4;
        if (ch < C) {
            const FT* fc = feat + ch;
            for (int bin = grp; bin < bins; bin += 4) {
                float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
                const Tap4* tp = s_tap + bin * spb;
#pragma unroll 4
                for (int sidx = 0; sidx < spb; ++sidx) {
                    const int4 of = *reinterpret_cast<const int4*>(&tp[sidx].o1);
                    const float4 w = *reinterpret_cast<const float4*>(&tp[sidx].w1);
                    const float4 v1 = ld4(fc + of.x), v2 = ld4(fc + of.y), v3 = ld4(fc + of.z), v4 = ld4(fc + of.w);
                    acc.x += ((w.x * v1.x + w.y * v2.x) + w.z * v3.x) + w.w * v4.x;
                    acc.y += ((w.x * v1.y + w.y * v2.y) + w.z * v3.y) + w.w * v4.y;
                    acc.z += ((w.x * v1.z + w.y * v2.z) + w.z * v3.z) + w.w * v4.z;
                    acc.w += ((w.x * v1.w + w.y * v2.w) + w.z * v3.w) + w.w * v4.w;
                }
                acc.x /= cnt; acc.y /= cnt; acc.z /= cnt; acc.w /= cnt;
                *reinterpret_cast<float4*>(&s_tile[bin * pitch + cq * 4]) = acc;
            }
        }
        __syncthreads();
        // out[r][c0 + cc][bin] is contiguous in (cc, bin): write it as 128-bit rows
        const int ctile = min(kCTile, C - c0);
        const int total = ctile * bins;
        float* dst = o + (long long)c0 * bins;
        if ((total & 3) == 0 && ((((long long)C * bins) & 3) == 0) && (((long long)c0 * bins) & 3) == 0) {
            for (int q = threadIdx.x; q < total / 4; q += blockDim.x) {
                float v[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int t = q * 4 + e;
                    const int cc = t / bins, bin = t - cc * bins;
                    v[e] = s_tile[bin * pitch + cc];
                }
                *reinterpret_cast<float4*>(dst + q * 4) = make_float4(v[0], v[1], v[2], v[3]);
            }
        } else {
            for (int t = threadIdx.x; t < total; t += blockDim.x) {
                const int cc = t / bins, bin = t - cc * bins;
                dst[t] = s_tile[bin * pitch + cc];
            }
        }
        __syncthreads();
    }
}


// ---- window kernel (2x2 samples per bin: every reference config) --------------------------------
// Design notes from the ncu captures of round 1 (profiles/):
//  * ptxas, left to its default occupancy target, sinks every tap load next to its use (2 loads
//    in flight per thread, 0.29 of the HBM roofline).  __launch_bounds__(NT, MINB) with a
//    register budget of ~80 makes it issue the whole window of a bin back-to-back.
//  * With the loads batched the kernel was bound by L1 wavefronts (784 128-bit taps per RoI per
//    4 channels), hence the tap de-duplication below; after that by the number of resident
//    warps (L1-miss latency x concurrency), hence 128-thread CTAs over 128 channels, 6 per SM.
// The 2x2 samples of a bin touch the cells {lo0, hi0, lo1, hi1} per axis.  With a sample
// spacing below two cells (RoI narrower than ~28 cells, i.e. every RoI the FPN level map
// sends to a level) lo1 - lo0 is 0, 1 or 2 and the taps fall into a (PY+2) x (PX+2) window of
// distinct cells, so a bin needs 4..16 loads instead of 16 (387 instead of 784 per RoI on the
// config-2 workload: the kernel was bound by L1 wavefronts, ncu prof_roi4).  The pattern
// (PY, PX) is uniform over the warps that share a bin, every sample still reads "its"
// four cells from the window registers and is summed in torchvision's order, so the result
// stays bit-identical to the reference.
struct __align__(16) BinTab {
    int ry[4];          // byte offsets of the window rows   (rows PY, PY+1 belong to sample iy = 1)
    int cx[4];          // byte offsets of the window columns
    float w[16];        // w1..w4 of the samples (iy, ix) = (0,0), (0,1), (1,0), (1,1)
    int pat, _p0, _p1, _p2;
};

// bf16 features (4 channels per lane, one 64-bit load per cell, converted to fp32): scalar additions
template <int PY, int PX>
__device__ __forceinline__ float4 bin_eval(const char* fb, const BinTab* t) {
    const int4 ry = *reinterpret_cast<const int4*>(t->ry);
    const int4 cx = *reinterpret_cast<const int4*>(t->cx);
    const int ryv[4] = {ry.x, ry.y, ry.z, ry.w}, cxv[4] = {cx.x, cx.y, cx.z, cx.w};
    float4 v[4][4];
#pragma unroll
    for (int r = 0; r < PY + 2; ++r) {
        const char* rp = fb + ryv[r];
#pragma unroll
        for (int c = 0; c < PX + 2; ++c) v[r][c] = ld4(reinterpret_cast<const __nv_bfloat16*>(rp + cxv[c]));
    }
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int iy = 0; iy < 2; ++iy) {
#pragma unroll
        for (int ix = 0; ix < 2; ++ix) {
            const int r0 = iy ? PY : 0, c0 = ix ? PX : 0;
            const float4 w = *reinterpret_cast<const float4*>(&t->w[(iy * 2 + ix) * 4]);
            const float4 &v1 = v[r0][c0], &v2 = v[r0][c0 + 1], &v3 = v[r0 + 1][c0], &v4 = v[r0 + 1][c0 + 1];
            // torchvision's order: ((w1 v1 + w2 v2) + w3 v3) + w4 v4, summed over samples
            acc.x += ((w.x * v1.x + w.y * v2.x) + w.z * v3.x) + w.w * v4.x;
            acc.y += ((w.x * v1.y + w.y * v2.y) + w.z * v3.y) + w.w * v4.y;
            acc.z += ((w.x * v1.z + w.y * v2.z) + w.z * v3.z) + w.w * v4.z;
            acc.w += ((w.x * v1.w + w.y * v2.w) + w.z * v3.w) + w.w * v4.w;
        }
    }
    return acc;
}

// fp32 features (4 channels per lane, one 128-bit load per cell): the same products and sums in the same order, with the
// additions two channels per instruction (add.rn.f32x2 -> FADD2).  The products stay scalar FMULs on purpose:
// ptxas (CUDA 12.9) contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 even with -fmad=false, which would change
// the rounding; a scalar product feeding a packed add is left alone (checked in SASS).
__device__ __forceinline__ unsigned long long add2(unsigned long long a, unsigned long long b) {
    unsigned long long r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ unsigned long long pack2(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
template <int PY, int PX>
__device__ __forceinline__ float4 bin_eval_x2(const char* fb, const BinTab* t) {
    const int4 ry = *reinterpret_cast<const int4*>(t->ry);
    const int4 cx = *reinterpret_cast<const int4*>(t->cx);
    const int ryv[4] = {ry.x, ry.y, ry.z, ry.w}, cxv[4] = {cx.x, cx.y, cx.z, cx.w};
    float4 v[4][4];
#pragma unroll
    for (int r = 0; r < PY + 2; ++r) {
        const char* rp = fb + (unsigned)ryv[r];      // offsets are non-negative: zero-extend, no sign shifts
#pragma unroll
        for (int c = 0; c < PX + 2; ++c) v[r][c] = __ldg(reinterpret_cast<const float4*>(rp + (unsigned)cxv[c]));
    }
    unsigned long long a01 = 0ull, a23 = 0ull;      // (+0, +0)
#pragma unroll
    for (int iy = 0; iy < 2; ++iy) {
#pragma unroll
        for (int ix = 0; ix < 2; ++ix) {
            const int r0 = iy ? PY : 0, c0 = ix ? PX : 0;
            const float4 w = *reinterpret_cast<const float4*>(&t->w[(iy * 2 + ix) * 4]);
            const float4 &v1 = v[r0][c0], &v2 = v[r0][c0 + 1], &v3 = v[r0 + 1][c0], &v4 = v[r0 + 1][c0 + 1];
            a01 = add2(a01, add2(add2(add2(pack2(w.x * v1.x, w.x * v1.y), pack2(w.y * v2.x, w.y * v2.y)),
                                      pack2(w.z * v3.x, w.z * v3.y)), pack2(w.w * v4.x, w.w * v4.y)));
            a23 = add2(a23, add2(add2(add2(pack2(w.x * v1.z, w.x * v1.w), pack2(w.y * v2.z, w.y * v2.w)),
                                      pack2(w.z * v3.z, w.z * v3.w)), pack2(w.w * v4.z, w.w * v4.w)));
        }
    }
    float4 acc;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(acc.x), "=f"(acc.y) : "l"(a01));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(acc.z), "=f"(acc.w) : "l"(a23));
    return acc;
}

__device__ __forceinline__ void sts_f32(unsigned addr, float v) {
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}

// NT threads per CTA, CT channels per CTA (grid.y = C / CT tiles), 4 channels per lane, MINB = min resident CTAs/SM
// (the register bound that keeps the window loads batched, see the notes above).
template <typename FT, int NT, int CT, int MINB>
__global__ void __launch_bounds__(NT, MINB) k_roi_align_win(RoiArgs a, float* __restrict__ out) {
    using Tab = BinTab;
    extern __shared__ __align__(16) float s_tile[];                      // [CT][bins] (+ bin table behind it)
    const long long r = blockIdx.x;
    const int tile = blockIdx.y;
    const b2d_roi_cfg& c = a.cfg;
    float x1, y1, x2, y2;
    int img;
    if (!roi_fetch(a, r, img, x1, y1, x2, y2)) return;
    int lvl;
    if (a.levels) lvl = a.levels[r];
    else lvl = c.num_levels > 1 ? roi_level(x1, y1, x2, y2, c.finest_scale, c.num_levels) : 0;
    const int H = c.H[lvl], W = c.W[lvl], C = c.C;
    const int bins = c.PH * c.PW;
    Tab* s_tab = reinterpret_cast<Tab*>(s_tile + CT * bins);
    const RoiGeom g = roi_geom(x1, y1, x2, y2, c.spatial_scale[lvl], c.PH, c.PW, 2, c.aligned);
    if ((int)threadIdx.x < bins) {
        const int bin = threadIdx.x, ph = bin / c.PW, pw = bin - ph * c.PW;
        const AxisTap ty0 = axis_tap(g.sy, g.bh, ph, 0, 2, H), ty1 = axis_tap(g.sy, g.bh, ph, 1, 2, H);
        const AxisTap tx0 = axis_tap(g.sx, g.bw, pw, 0, 2, W), tx1 = axis_tap(g.sx, g.bw, pw, 1, 2, W);
        const int es = (int)sizeof(FT);
        Tab t;
        // window rows: PY in {0,1}: lo0 + {0..PY+1} clamped like the taps; PY = 2: {lo0, hi0, lo1, hi1}
        const int dy = ty1.lo - ty0.lo, dx = tx1.lo - tx0.lo;
        const int py = (dy >= 0 && dy < 2) ? dy : 2, px = (dx >= 0 && dx < 2) ? dx : 2;   // 2 = explicit {lo0,hi0,lo1,hi1}
        int yy[4], xx[4];
        if (py < 2) { for (int k = 0; k < 4; ++k) yy[k] = min(ty0.lo + k, H - 1); }
        else { yy[0] = ty0.lo; yy[1] = ty0.hi; yy[2] = ty1.lo; yy[3] = ty1.hi; }
        if (px < 2) { for (int k = 0; k < 4; ++k) xx[k] = min(tx0.lo + k, W - 1); }
        else { xx[0] = tx0.lo; xx[1] = tx0.hi; xx[2] = tx1.lo; xx[3] = tx1.hi; }
        for (int k = 0; k < 4; ++k) { t.ry[k] = yy[k] * W * C * es; t.cx[k] = xx[k] * C * es; }
        const AxisTap* tys[2] = {&ty0, &ty1};
        const AxisTap* txs[2] = {&tx0, &tx1};
        for (int iy = 0; iy < 2; ++iy)
            for (int ix = 0; ix < 2; ++ix) {
                const AxisTap& ty = *tys[iy];
                const AxisTap& tx = *txs[ix];
                const bool ok = ty.valid && tx.valid;
                const float wv[4] = {ok ? ty.h * tx.h : 0.0f, ok ? ty.h * tx.l : 0.0f, ok ? ty.l * tx.h : 0.0f,
                                     ok ? ty.l * tx.l : 0.0f};
                for (int k = 0; k < 4; ++k) t.w[(iy * 2 + ix) * 4 + k] = wv[k];
            }
        t.pat = py * 3 + px; t._p0 = t._p1 = t._p2 = 0;
        s_tab[bin] = t;
    } else if ((int)threadIdx.x >= NT - 16) {           // byte offsets of the rotated tile stores: [rot][step]
        const int k = threadIdx.x - (NT - 16);
        reinterpret_cast<int*>(s_tab + bins)[k] = (((k & 3) + (k >> 2)) & 3) * bins * 4;
    }
    __syncthreads();
    const FT* feat = reinterpret_cast<const FT*>(a.feat[lvl]) + (long long)img * H * W * C;
    constexpr int LG = CT / 4, NG = NT / LG;               // lanes per bin group, bin groups
    const int cq = threadIdx.x % LG, grp = threadIdx.x / LG;
    float* o = out + r * (long long)C * bins;
    {
        const int c0 = tile * CT;
        const int ch = c0 + cq * 4;
        if (ch < C) {
            const char* fb = reinterpret_cast<const char*>(feat + ch);
            // The lanes of a warp are 4 * bins floats apart in the [channel][bin] tile, i.e. on 8 banks only; lane
            // group j = cq / 8 therefore stores component (s + j) % 4 at step s, which spreads every store over
            // all 32 banks (bins odd).  The rotation is two rounds of selects on the results.
            // Their four tile offsets come from a 16-entry table in shared memory (one LDS.128 per bin) so that
            // they occupy no registers while the window is live.
            const int rot = (cq >> 3) & 3;
            const bool r1 = rot & 1, r2 = rot & 2;
            const int4* s_rot = reinterpret_cast<const int4*>(s_tab + bins) + rot;
            const unsigned st_base = (unsigned)__cvta_generic_to_shared(s_tile + (cq * 4) * bins);
            for (int bin = grp; bin < bins; bin += NG) {
                const Tab* t = s_tab + bin;
                float4 acc;
                const int pat = t->pat, py = pat / 3, px = pat - py * 3;   // uniform over the warps of a bin
#define B2D_BIN(PY_, PX_)                                                  \
    do {                                                                   \
        if constexpr (sizeof(FT) == 4) acc = bin_eval_x2<PY_, PX_>(fb, t); \
        else acc = bin_eval<PY_, PX_>(fb, t);                              \
    } while (0)
                if (py == 0) {
                    if (px == 0) B2D_BIN(0, 0);
                    else if (px == 1) B2D_BIN(0, 1);
                    else B2D_BIN(0, 2);
                } else if (py == 1) {
                    if (px == 0) B2D_BIN(1, 0);
                    else if (px == 1) B2D_BIN(1, 1);
                    else B2D_BIN(1, 2);
                } else {
                    if (px == 0) B2D_BIN(2, 0);
                    else if (px == 1) B2D_BIN(2, 1);
                    else B2D_BIN(2, 2);
                }
#undef B2D_BIN
                // x / 4 == x * 0.25 exactly; rotated stores, see the rotation note above
                const float f0 = acc.x * 0.25f, f1 = acc.y * 0.25f, f2 = acc.z * 0.25f, f3 = acc.w * 0.25f;
                const float g0 = r1 ? f1 : f0, g1 = r1 ? f2 : f1, g2 = r1 ? f3 : f2, g3 = r1 ? f0 : f3;
                const int4 ro = *s_rot;
                const unsigned sb = st_base + bin * 4;
                sts_f32(sb + ro.x, r2 ? g2 : g0);       // f[(s + rot) % 4] at step s
                sts_f32(sb + ro.y, r2 ? g3 : g1);
                sts_f32(sb + ro.z, r2 ? g0 : g2);
                sts_f32(sb + ro.w, r2 ? g1 : g3);
            }
        }
        // the [ctile][bins] tile is contiguous in shared memory and in HBM: ONE bulk async store (TMA engine) instead
        // of an LDS.128 + STG.128 per 16 bytes through the LSU pipe, which this kernel keeps 64 % busy (ncu r1j).
        // C % 4 == 0 (checked by the launcher) makes its size and its offset in the output multiples of 16 bytes.
        const int ctile = min(CT, C - c0);
        const int total = ctile * bins;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncthreads();
        if (threadIdx.x == 0) {
            const unsigned src = (unsigned)__cvta_generic_to_shared(s_tile);
            float* dstp = o + (long long)c0 * bins;
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dstp), "r"(src), "r"((unsigned)(total * 4)) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        }
    }
}

// ---- NCHW -> NHWC (fp32): lets reference-layout features (lib/necks.py FPN output) use the
// channel-vectorised kernels above.  64(hw) x 32(c) tiles through padded shared memory; reads
// are 256 B runs along hw, writes 128 B runs along c.
__global__ void __launch_bounds__(256) k_nchw_to_nhwc(float* __restrict__ dst, const float* __restrict__ src, int C,
                                                      long long HW) {
    __shared__ float tile[32][65];
    const long long b = blockIdx.z;
    const float* s = src + b * C * HW;
    float* d = dst + b * C * HW;
    const long long hw0 = (long long)blockIdx.x * 64;
    const int c0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;       // 64 x 4
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int c = c0 + ty + 4 * k;
        const long long hw = hw0 + tx;
        if (c < C && hw < HW) tile[ty + 4 * k][tx] = s[(long long)c * HW + hw];
    }
    __syncthreads();
    const int cx = threadIdx.x & 31, hy = threadIdx.x >> 5;       // 32 x 8
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const long long hw = hw0 + hy + 8 * k;
        const int c = c0 + cx;
        if (c < C && hw < HW) d[hw * C + c] = tile[cx][hy + 8 * k];
    }
}

// generic: one thread per output element (r, c, ph, pw); layout 0 = NCHW fp32, 1 = NHWC fp32
__global__ void __launch_bounds__(256) k_roi_align_any(RoiArgs a, float* __restrict__ out) {
    const b2d_roi_cfg& c = a.cfg;
    const int bins = c.PH * c.PW;
    const long long total = a.R * c.C * bins;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const int pw = (int)(t % c.PW), ph = (int)((t / c.PW) % c.PH);
    const int ch = (int)((t / bins) % c.C);
    const long long r = t / ((long long)bins * c.C);
    float x1, y1, x2, y2;
    int img;
    if (!roi_fetch(a, r, img, x1, y1, x2, y2)) return;
    int lvl;
    if (a.levels) lvl = a.levels[r];
    else lvl = c.num_levels > 1 ? roi_level(x1, y1, x2, y2, c.finest_scale, c.num_levels) : 0;
    const int H = c.H[lvl], W = c.W[lvl];
    const RoiGeom g = roi_geom(x1, y1, x2, y2, c.spatial_scale[lvl], c.PH, c.PW, c.sampling_ratio, c.aligned);
    const float* f = reinterpret_cast<const float*>(a.feat[lvl]);
    long long sy, sx, base;
    if (c.layout == 0) { base = ((long long)img * c.C + ch) * H * W; sy = W; sx = 1; }
    else { base = (long long)img * H * W * c.C + ch; sy = (long long)W * c.C; sx = c.C; }
    float acc = 0.0f;
    for (int iy = 0; iy < g.gy; ++iy) {
        const AxisTap ty = axis_tap(g.sy, g.bh, ph, iy, g.gy, H);
        for (int ix = 0; ix < g.gx; ++ix) {
            const AxisTap tx = axis_tap(g.sx, g.bw, pw, ix, g.gx, W);
            if (!(ty.valid && tx.valid)) continue;
            const float v1 = __ldg(f + base + ty.lo * sy + tx.lo * sx), v2 = __ldg(f + base + ty.lo * sy + tx.hi * sx);
            const float v3 = __ldg(f + base + ty.hi * sy + tx.lo * sx), v4 = __ldg(f + base + ty.hi * sy + tx.hi * sx);
            const float w1 = ty.h * tx.h, w2 = ty.h * tx.l, w3 = ty.l * tx.h, w4 = ty.l * tx.l;
            acc += ((w1 * v1 + w2 * v2) + w3 * v3) + w4 * v4;
        }
    }
    out[t] = acc / (float)max(g.gy * g.gx, 1);
}

}  // namespace b2d

using namespace b2d;

extern "C" {

int b2d_roi_levels(int* levels, const float* rois, long long roi_ld, long long R, float finest_scale,
                   int num_levels, void* stream) {
    B2D_REQUIRE(levels && rois && R >= 0 && num_levels >= 1, "roi_levels: bad args");
    if (R == 0) return B2D_OK;
    k_roi_levels<<<cdiv(R, 256), 256, 0, (cudaStream_t)stream>>>(levels, rois, roi_ld, R, finest_scale, num_levels);
    return check_launch("roi_levels");
}

static int roi_align_launch(float* out, const void* const* feat_ptrs_host, const float* rois, long long roi_ld,
                            const int* roi_img, const int* levels, long long R, long long batched_ld,
                            const int* counts, const b2d_roi_cfg* cfg_host, void* stream) {
    B2D_REQUIRE(out && feat_ptrs_host && rois && cfg_host && R >= 0, "roi_align_fwd: bad args");
    const b2d_roi_cfg& c = *cfg_host;
    B2D_REQUIRE(c.num_levels >= 1 && c.num_levels <= B2D_MAX_LEVELS && c.C >= 1 && c.PH >= 1 && c.PW >= 1,
                "roi_align_fwd: bad cfg");
    B2D_REQUIRE(c.layout >= 0 && c.layout <= 2, "roi_align_fwd: layout must be 0 (NCHW), 1 (NHWC) or 2 (NHWC bf16)");
    if (R == 0) return B2D_OK;
    RoiArgs a;
    memset(&a, 0, sizeof(a));
    a.cfg = c;
    for (int l = 0; l < c.num_levels; ++l) a.feat[l] = feat_ptrs_host[l];
    a.rois = rois; a.roi_ld = roi_ld; a.roi_img = roi_img; a.levels = levels; a.R = R;
    a.batched_ld = batched_ld; a.counts = counts;
    cudaStream_t st = (cudaStream_t)stream;
    const int bins = c.PH * c.PW;
    const bool fast = c.layout >= 1 && c.sampling_ratio > 0 &&
                      bins * c.sampling_ratio * c.sampling_ratio <= kMaxSamples && (c.C % 4) == 0 &&
                      bins * (kCTile + 4) * 4 <= 200 * 1024;
    // 2x2 samples per bin (every reference config): window kernel, 128 channels per 128-thread CTA
    const bool win = fast && c.sampling_ratio == 2 && bins <= 64;
    if (win) {
        int rc5 = 0;
        auto launch5 = [&](auto kern, int nt, int ct) {
            const size_t smem5 = (size_t)ct * bins * 4 + (size_t)bins * sizeof(BinTab) + 64;
            if ((rc5 = set_dyn_smem(kern, smem5, "k_roi_align_win")) != 0) return;
            kern<<<dim3((unsigned)R, (unsigned)cdiv(c.C, ct)), nt, smem5, st>>>(a, out);
        };
        // 128 threads x 4 channels = 128 channels per CTA, 6 CTAs/SM: fastest of the measured
        // (threads, channels/CTA, CTAs/SM, channels/thread) points -- (256,256,2,4) 200 us,
        // (256,256,3,4) 169, (128,128,4,4) 169, (128,128,6,4) 159, (128,128,7,4) 186 (spills),
        // (256,128,5,2) 175, (128,64,8,2) 186, (128,64,10,2) 173 (config 2, 4096 RoIs)
        if (c.layout == 1) launch5(k_roi_align_win<float, 128, 128, 6>, 128, 128);
        else launch5(k_roi_align_win<__nv_bfloat16, 128, 128, 6>, 128, 128);
        if (rc5) return rc5;
    } else if (fast) {
        const size_t smem = (size_t)bins * (kCTile + 4) * 4;
        if (c.layout == 1) {
            B2D_SMEM(k_roi_align_nhwc<float>, smem, "k_roi_align_nhwc");   // per device
            k_roi_align_nhwc<float><<<(unsigned)R, 256, smem, st>>>(a, out);
        } else {
            B2D_SMEM(k_roi_align_nhwc<__nv_bfloat16>, smem, "k_roi_align_nhwc");
            k_roi_align_nhwc<__nv_bfloat16><<<(unsigned)R, 256, smem, st>>>(a, out);
        }
    } else {
        B2D_REQUIRE(c.layout != 2, "roi_align_fwd: bf16 needs NHWC, C % 4 == 0 and a fixed sampling_ratio");
        const long long total = R * c.C * bins;
        k_roi_align_any<<<cdiv(total, 256), 256, 0, st>>>(a, out);
    }
    return check_launch("roi_align_fwd");
}

int b2d_roi_align_fwd(float* out, const void* const* feat_ptrs_host, const float* rois, long long roi_ld,
                      const int* roi_img, const int* levels, long long R, const b2d_roi_cfg* cfg_host,
                      void* stream) {
    return roi_align_launch(out, feat_ptrs_host, rois, roi_ld, roi_img, levels, R, 0, nullptr, cfg_host, stream);
}

int b2d_roi_align_fwd_batched(float* out, const void* const* feat_ptrs_host, const float* rois, long long ld,
                              const int* counts, int B, const b2d_roi_cfg* cfg_host, void* stream) {
    B2D_REQUIRE(counts && ld >= 1 && B >= 1, "roi_align_fwd_batched: bad args");
    return roi_align_launch(out, feat_ptrs_host, rois, ld, nullptr, nullptr, (long long)B * ld, ld, counts, cfg_host,
                            stream);
}

int b2d_nchw_to_nhwc(float* dst, const float* src, int B, int C, int H, int W, void* stream) {
    B2D_REQUIRE(dst && src && B >= 1 && C >= 1 && H >= 1 && W >= 1, "nchw_to_nhwc: bad args");
    const long long HW = (long long)H * W;
    B2D_REQUIRE(cdiv(C, 32) <= 65535 && B <= 65535, "nchw_to_nhwc: C or B too large");
    dim3 grid(cdiv(HW, 64), cdiv(C, 32), B);
    k_nchw_to_nhwc<<<grid, 256, 0, (cudaStream_t)stream>>>(dst, src, C, HW);
    return check_launch("nchw_to_nhwc");
}

}  // extern "C"
