// common.cuh -- shared device/host helpers for the b200det kernels (sm_100a).
//
// Numerics contract: the whole library is compiled with -fmad=false and without
// --use_fast_math, so every fp32 +,-,*,/ rounds individually (IEEE, RN) in the
// order written -- the property the bit-exact parity with the reference's torch
// expressions rests on (SURVEY 7 "Bit-exact fp32 IoU/labels").
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/b200det.h"

namespace b2d {

constexpr int kMaxLevels = B2D_MAX_LEVELS;
constexpr int kMaxAnchorsPerCell = B2D_MAX_ANCHORS;

void set_error(const char* msg);
int check_launch(const char* what);

// Development knobs (DESIGN.md "Development knobs").  Read from the environment ONCE, when the library is first used
// (b2d_reload_knobs() re-reads them: tests only) -- no launcher calls getenv on the hot path.
struct Knobs {
    int dbg;               // B2D_DBG            select.cu debug switch
    int rpn_chains;        // B2D_RPN_CHAINS     1: per-level chains on internal streams (multi-kernel path)
    int rpn_front;         // B2D_RPN_FRONT      1: cluster kernel k_rpn_front (hist + threshold + compact + sort + decode)
    int rpn_back;          // B2D_RPN_BACK       1: cluster kernel k_rpn_back (cut + sweep + scan + merge)
    double nms_cut;        // B2D_NMS_CUT        score-cut factor (default 1.5), 0 disables
    int nms_p1_chains;     // B2D_NMS_P1_CHAINS
    int nms_sweep;         // B2D_NMS_SWEEP      0 disables the x-sweep mask kernel
    int sweep_t, sweep_g;  // B2D_SWEEP_T / _G   launch shape of k_nms_sweep
    int roi_bwd_tile;      // B2D_ROI_BWD_TILE   2: patch form (default), 1: tile-gather form, 0: generic backward kernel
    int assign_old;        // B2D_ASSIGN_OLD     1: round-1a assignment kernels in pyramid mode
    int debug_sync;        // B2D_DEBUG_SYNC     synchronise after every launch (localise a faulting kernel)
    int sample_threads;    // B2D_SAMPLE_THREADS 128 / 256: slim k_sample CTAs (default 1024)
    int pdl;               // B2D_PDL            1: programmatic dependent launch edges front -> back -> RoI targets (default 0)
};
const Knobs& knobs();

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) with its return code checked (set on every call: it is per device)
template <typename K>
inline int set_dyn_smem(K kern, size_t bytes, const char* what) {
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) return 0;
    char buf[256];
    snprintf(buf, sizeof(buf), "%s: cudaFuncSetAttribute(%zu B of dynamic shared memory): %s", what, bytes, cudaGetErrorString(e));
    b2d::set_error(buf);
    (void)cudaGetLastError();
    return (int)e;
}
#define B2D_SMEM(kern, bytes, what)                          \
    do {                                                     \
        const int rc_ = b2d::set_dyn_smem(kern, bytes, what); \
        if (rc_) return rc_;                                 \
    } while (0)

// Programmatic dependent launch (sm_90+): a kernel launched with cudaLaunchAttributeProgrammaticStreamSerialization may
// become resident while its stream predecessor still runs, once every CTA of the predecessor has executed
// pdl_launch_dependents() (or exited); pdl_wait() blocks until the predecessor has COMPLETED and its writes are visible.
// Both are no-ops for a kernel that was launched the ordinary way.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

#define B2D_REQUIRE(cond, msg)            \
    do {                                  \
        if (!(cond)) {                    \
            b2d::set_error(msg);          \
            return B2D_ERR_ARG;           \
        }                                 \
    } while (0)

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

// ---- monotone float <-> uint key (larger float => larger key; total order) ----
__host__ __device__ __forceinline__ uint32_t f2key(float f) {
    // -0.0 and +0.0 compare equal (torch.topk / sort treat them as one value and order the tie by index): one key for
    // both, else a -0.0 logit would rank below a +0.0 one of a higher index
    f = f + 0.0f;
#ifdef __CUDA_ARCH__
    uint32_t u = __float_as_uint(f);
#else
    union { float f; uint32_t u; } c; c.f = f; uint32_t u = c.u;
#endif
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ __forceinline__ float key2f(uint32_t k) {
    uint32_t u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
#ifdef __CUDA_ARCH__
    return __uint_as_float(u);
#else
    union { float f; uint32_t u; } c; c.u = u; return c.f;
#endif
}

// composite sort key: (score key, lowest index first) -> all composites distinct,
// "descending composite" == "descending score, ties by ascending index".
__device__ __forceinline__ uint64_t make_comp(uint32_t key, uint32_t idx) {
    return ((uint64_t)key << 32) | (uint64_t)(0xffffffffu - idx);
}
__device__ __forceinline__ uint32_t comp_key(uint64_t c) { return (uint32_t)(c >> 32); }
__device__ __forceinline__ uint32_t comp_idx(uint64_t c) { return 0xffffffffu - (uint32_t)c; }

// ---- exact reference arithmetic -------------------------------------------------
struct Box { float x1, y1, x2, y2; };

// lib/utils.py:151-172 (calc_iou): +1 areas, strict tl<br mask applied as a multiply
// (keeps the reference's signed zeros), one IEEE divide.  aa/ab = precomputed +1 areas.
__device__ __forceinline__ float iou_plus1(const Box& a, float aa, const Box& b, float ab) {
    const float tlx = fmaxf(a.x1, b.x1), tly = fmaxf(a.y1, b.y1);
    const float brx = fminf(a.x2, b.x2), bry = fminf(a.y2, b.y2);
    const float dx = (brx - tlx) + 1.0f, dy = (bry - tly) + 1.0f;
    const bool hit = (tlx < brx) && (tly < bry);
    const float ai = (dx * dy) * (hit ? 1.0f : 0.0f);
    const float s = aa + ab;
    // miss & positive union: (+-0)/s == +-0 == ai, no divide needed (94% of RPN pairs)
    if (!hit && s > 0.0f) return ai;
    return ai / (s - ai);
}
__device__ __forceinline__ float area_plus1(const Box& b) {
    return ((b.x2 - b.x1) + 1.0f) * ((b.y2 - b.y1) + 1.0f);
}

// lib/utils.py:83-92,134-144,109-120: param2bbox (+ optional clamp)
__device__ __forceinline__ Box decode_box(const Box& base, float p0, float p1, float p2, float p3,
                                          const float* __restrict__ ms /*means[4], stds[4]*/,
                                          bool clamp, float img_h, float img_w) {
    const float bw = (base.x2 - base.x1) + 1.0f, bh = (base.y2 - base.y1) + 1.0f;
    const float bcx = (base.x2 + base.x1) / 2.0f, bcy = (base.y2 + base.y1) / 2.0f;
    const float tx = p0 * ms[4] + ms[0], ty = p1 * ms[5] + ms[1];
    const float tw = p2 * ms[6] + ms[2], th = p3 * ms[7] + ms[3];
    const float cx = tx * bw + bcx, cy = ty * bh + bcy;
    const float w = expf(tw) * bw, h = expf(th) * bh;
    Box o;
    o.x1 = cx - w / 2.0f; o.y1 = cy - h / 2.0f; o.x2 = cx + w / 2.0f; o.y2 = cy + h / 2.0f;
    if (clamp) {
        const float mx = img_w - 1.0f, my = img_h - 1.0f;
        o.x1 = fminf(fmaxf(o.x1, 0.0f), mx); o.x2 = fminf(fmaxf(o.x2, 0.0f), mx);
        o.y1 = fminf(fmaxf(o.y1, 0.0f), my); o.y2 = fminf(fmaxf(o.y2, 0.0f), my);
    }
    return o;
}

// lib/anchor.py:107-129: anchor (a, y, x) of one level, computed in registers.
__device__ __forceinline__ Box anchor_at(const b2d_level& lv, int a, int y, int x) {
    float cx = (float)x * lv.stride, cy = (float)y * lv.stride;
    if (!lv.center_lt) { cx = cx + lv.stride / 2.0f; cy = cy + lv.stride / 2.0f; }
    const float hw = lv.ws[a] / 2.0f, hh = lv.hs[a] / 2.0f;
    Box b; b.x1 = cx - hw; b.y1 = cy - hh; b.x2 = cx + hw; b.y2 = cy + hh;
    return b;
}
__device__ __forceinline__ Box anchor_flat(const b2d_level& lv, int i) {
    const int hw = lv.H * lv.W;
    const int a = i / hw, r = i - a * hw;
    const int y = r / lv.W, x = r - y * lv.W;
    return anchor_at(lv, a, y, x);
}

// ---- warp helpers ---------------------------------------------------------------
__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

// warp-aggregated slot allocation: returns this lane's slot (valid only if pred)
__device__ __forceinline__ int warp_alloc(bool pred, int* counter) {
    const unsigned m = __ballot_sync(0xffffffffu, pred);
    if (m == 0) return -1;
    const int leader = __ffs(m) - 1;
    int base = 0;
    if (lane_id() == leader) base = atomicAdd(counter, __popc(m));
    base = __shfl_sync(0xffffffffu, base, leader);
    return base + __popc(m & ((1u << lane_id()) - 1u));
}

// 64-bit mix (splitmix64 finaliser) -> 32-bit sampling key; part of the device-RNG
// sampler spec (DESIGN.md "Samplers"), restated by oracle/sampler_spec.py.
__host__ __device__ __forceinline__ uint32_t mix_key(uint64_t seed, uint64_t i) {
    uint64_t z = seed + 0x9E3779B97F4A7C15ull * (i + 1);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z = z ^ (z >> 31);
    return (uint32_t)(z >> 32);
}

// ---- block-wide bitonic sort of u64 keys, DESCENDING ---------------------------------
// n = E * blockDim.x keys live in s[0..n).  Each thread keeps E consecutive keys in
// registers: strides < E are compare-exchanges inside the thread, strides < 32*E are warp
// shuffles, and only strides >= 32*E go through shared memory (conflict-free [e][thread]
// layout) -- 15 shared-memory exchanges instead of 78 barrier-separated passes for n = 4096.
__device__ __forceinline__ uint64_t shfl_xor_u64(uint64_t v, int m) {
    const uint32_t lo = __shfl_xor_sync(0xffffffffu, (uint32_t)v, m);
    const uint32_t hi = __shfl_xor_sync(0xffffffffu, (uint32_t)(v >> 32), m);
    return ((uint64_t)hi << 32) | lo;
}

template <int E>
__device__ __forceinline__ void block_sort_desc_E(uint64_t* s) {
    const int t = threadIdx.x, T = blockDim.x;
    const int n = E * T;
    uint64_t v[E];
#pragma unroll
    for (int e = 0; e < E; ++e) v[e] = s[t * E + e];
    for (int k = 2; k <= n; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            if (j >= 32 * E) {
                __syncthreads();
#pragma unroll
                for (int e = 0; e < E; ++e) s[e * T + t] = v[e];
                __syncthreads();
                const int pt = t ^ (j / E);
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    const int x = t * E + e;
                    const uint64_t o = s[e * T + pt];
                    const bool want_max = (((x & j) == 0) == ((x & k) == 0));
                    v[e] = want_max ? (v[e] > o ? v[e] : o) : (v[e] < o ? v[e] : o);
                }
            } else if (j >= E) {
                const int m = j / E;
#pragma unroll
                for (int e = 0; e < E; ++e) {
                    const int x = t * E + e;
                    const uint64_t o = shfl_xor_u64(v[e], m);
                    const bool want_max = (((x & j) == 0) == ((x & k) == 0));
                    v[e] = want_max ? (v[e] > o ? v[e] : o) : (v[e] < o ? v[e] : o);
                }
            } else {
#pragma unroll
                for (int jj = E / 2; jj > 0; jj >>= 1) {
                    if (jj != j) continue;
#pragma unroll
                    for (int e = 0; e < E; ++e) {
                        if (e & jj) continue;
                        const int x = t * E + e;
                        const bool desc = ((x & k) == 0);
                        const uint64_t a = v[e], b = v[e | jj];
                        if ((a < b) == desc) { v[e] = b; v[e | jj] = a; }
                    }
                }
            }
        }
    }
    __syncthreads();
#pragma unroll
    for (int e = 0; e < E; ++e) s[t * E + e] = v[e];
    __syncthreads();
}

// Sort s[0..n) descending; n must be a power of two, entries [n, max(n, blockDim)) must be
// writable (they are zero-filled here).  blockDim.x must be 1024.
__device__ __forceinline__ void bitonic_sort_desc(uint64_t* s, int n) {
    const int T = blockDim.x;
    if (n < T) {
        for (int i = n + threadIdx.x; i < T; i += T) s[i] = 0ull;
        n = T;
    }
    __syncthreads();
    switch (n / T) {
        case 1: block_sort_desc_E<1>(s); break;
        case 2: block_sort_desc_E<2>(s); break;
        case 4: block_sort_desc_E<4>(s); break;
        case 8: block_sort_desc_E<8>(s); break;
        default: block_sort_desc_E<16>(s); break;
    }
}

}  // namespace b2d
