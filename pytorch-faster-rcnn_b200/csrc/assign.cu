// assign.cu -- K2: tiled pairwise IoU with fused row max/argmax assignment and the
// per-GT best-anchor rule of MaxIoUAssigner (lib/region.py:75-107), batched over
// images, with anchors generated in registers (no [4,N] anchor tensor and no
// [N,K] IoU table ever touch HBM).  Plus the label census, the device-RNG sampler
// (a5) and the fused target gather/encode (a6/a13 + K8).
//
// Roofline: HBM-bound on its 12 B/anchor output (int64 label + fp32 IoU) for the
// handful of GTs of config 2; fp32-issue bound beyond K ~ 8 (SURVEY 8(d)).
#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "targets_common.cuh"

namespace b2d {

// (in_h, in_w) of inside_grid_mask (lib/region.py:11-13): python float64 reciprocal multiply
__device__ __forceinline__ void grid_limits(const b2d_level& lv, float img_h, float img_w, int& in_h, int& in_w) {
    const double r = 1.0 / (double)lv.stride;
    in_h = min(lv.H, (int)((double)img_h * r) + 1);
    in_w = min(lv.W, (int)((double)img_w * r) + 1);
}

// Fetch box i of image b (explicit or generated); returns false if it is masked out.
__device__ __forceinline__ bool load_box(const AssignArgs& p, const b2d_pyramid& pyr, int b, long long i,
                                         long long n_b, Box& bx, const int* __restrict__ s_lim) {
    if (i >= n_b) return false;
    if (!p.use_pyr) {
        const float* src = p.boxes + (long long)b * 4 * p.box_ld;
        bx.x1 = src[i]; bx.y1 = src[p.box_ld + i]; bx.x2 = src[2 * p.box_ld + i]; bx.y2 = src[3 * p.box_ld + i];
        return true;
    }
    int l = 0;
#pragma unroll
    for (int q = 1; q < kMaxLevels; ++q)
        if (q < pyr.num_levels && i >= pyr.lv[q].offset) l = q;
    const b2d_level& lv = pyr.lv[l];
    const int li = (int)(i - lv.offset);
    const int hw = lv.H * lv.W;
    const int a = li / hw, r = li - a * hw;
    const int y = r / lv.W, x = r - y * lv.W;
    bx = anchor_at(lv, a, y, x);
    const float img_h = p.img_hw[2 * b], img_w = p.img_hw[2 * b + 1];
    bool ok = (y < s_lim[2 * l]) && (x < s_lim[2 * l + 1]);
    if (p.border >= 0.0f)
        ok = ok && bx.x1 >= -p.border && bx.y1 >= -p.border && bx.x2 < img_w + p.border && bx.y2 < img_h + p.border;
    return ok;
}

// ---- pass 1: per-GT column max over all (valid) boxes  (lib/region.py:86) ------
__global__ void __launch_bounds__(256) k_assign_colmax(AssignArgs p, b2d_pyramid pyr, uint32_t* __restrict__ colmax) {
    __shared__ Box s_gt[kGtChunk];
    __shared__ float s_ga[kGtChunk];
    __shared__ uint32_t s_max[kGtChunk];
    const int b = blockIdx.y;
    const int K = p.gt_count[b];
    const long long n_b = p.box_count ? (long long)p.box_count[b] : p.N;
    const float* g = p.gt + (long long)b * 4 * p.gt_ld;
    const uint32_t kNegInf = f2key(-INFINITY), kZero = f2key(0.0f);
    __shared__ int s_lim[2 * kMaxLevels];
    if (p.use_pyr && threadIdx.x < pyr.num_levels)     // fp64 once per (block, level), not per box
        grid_limits(pyr.lv[threadIdx.x], p.img_hw[2 * b], p.img_hw[2 * b + 1], s_lim[2 * threadIdx.x], s_lim[2 * threadIdx.x + 1]);
    __syncthreads();

    Box bx[kBoxesPerThread];
    float ba[kBoxesPerThread];
    bool ok[kBoxesPerThread];
    const long long base = ((long long)blockIdx.x * blockDim.x) * kBoxesPerThread + threadIdx.x;
#pragma unroll
    for (int r = 0; r < kBoxesPerThread; ++r) {
        ok[r] = load_box(p, pyr, b, base + (long long)r * blockDim.x, n_b, bx[r], s_lim);
        ba[r] = ok[r] ? area_plus1(bx[r]) : 0.0f;
    }
    bool any_ok = false;
#pragma unroll
    for (int r = 0; r < kBoxesPerThread; ++r) any_ok |= ok[r];
    any_ok = __any_sync(0xffffffffu, any_ok);          // warp-uniform
    for (int j0 = 0; j0 < K; j0 += kGtChunk) {
        const int kc = min(kGtChunk, K - j0);
        __syncthreads();
        for (int j = threadIdx.x; j < kc; j += blockDim.x) {
            Box t{g[j0 + j], g[p.gt_ld + j0 + j], g[2 * p.gt_ld + j0 + j], g[3 * p.gt_ld + j0 + j]};
            s_gt[j] = t; s_ga[j] = area_plus1(t); s_max[j] = kNegInf;
        }
        __syncthreads();
        for (int j = 0; j < kc; ++j) {
            const Box t = s_gt[j];
            const float ta = s_ga[j];
            uint32_t m = any_ok ? kZero : kNegInf;      // every valid box contributes at least +-0
#pragma unroll
            for (int r = 0; r < kBoxesPerThread; ++r) {
                if (!ok[r]) continue;
                // a miss with positive areas is +-0 (see iou_plus1): only hits need arithmetic
                const bool hit = fmaxf(bx[r].x1, t.x1) < fminf(bx[r].x2, t.x2) && fmaxf(bx[r].y1, t.y1) < fminf(bx[r].y2, t.y2);
                if (hit || !(ba[r] > 0.0f && ta > 0.0f)) {
                    const float v = iou_plus1(bx[r], ba[r], t, ta) + 0.0f;  // -0 -> +0
                    m = max(m, f2key(v));
                }
            }
            if (__any_sync(0xffffffffu, m > kZero) || j0 + j == 0 || !any_ok) {
                m = __reduce_max_sync(0xffffffffu, m);
                if (lane_id() == 0 && m > s_max[j]) atomicMax(&s_max[j], m);
            } else if (lane_id() == 0 && s_max[j] < kZero) {
                atomicMax(&s_max[j], kZero);
            }
        }
        __syncthreads();
        for (int j = threadIdx.x; j < kc; j += blockDim.x)
            if (s_max[j] != kNegInf) atomicMax(&colmax[(long long)b * p.gt_ld + j0 + j], s_max[j]);
    }
}

// ---- pass 2: labels + IoU of the assigned GT + census  (lib/region.py:88-107) ---
__global__ void __launch_bounds__(256) k_assign_label(AssignArgs p, b2d_pyramid pyr,
                                                      const uint32_t* __restrict__ colmax,
                                                      int64_t* __restrict__ labels, float* __restrict__ out_iou,
                                                      int* __restrict__ census, int* __restrict__ pos_list,
                                                      int pos_cap) {
    __shared__ Box s_gt[kGtChunk];
    __shared__ float s_ga[kGtChunk];
    __shared__ float s_cm[kGtChunk];
    __shared__ int s_cnt[2];
    const int b = blockIdx.y;
    const int K = p.gt_count[b];
    const long long n_b = p.box_count ? (long long)p.box_count[b] : p.N;
    const float* g = p.gt + (long long)b * 4 * p.gt_ld;
    const int lead = p.prepend_gt ? K : 0;
    if (threadIdx.x < 2) s_cnt[threadIdx.x] = 0;
    __shared__ int s_lim[2 * kMaxLevels];
    if (p.use_pyr && threadIdx.x < pyr.num_levels)
        grid_limits(pyr.lv[threadIdx.x], p.img_hw[2 * b], p.img_hw[2 * b + 1], s_lim[2 * threadIdx.x], s_lim[2 * threadIdx.x + 1]);
    __syncthreads();

    Box bx[kBoxesPerThread];
    float ba[kBoxesPerThread], best[kBoxesPerThread], veq[kBoxesPerThread];
    int arg[kBoxesPerThread], eq[kBoxesPerThread];
    bool ok[kBoxesPerThread];
    const long long base = ((long long)blockIdx.x * blockDim.x) * kBoxesPerThread + threadIdx.x;
#pragma unroll
    for (int r = 0; r < kBoxesPerThread; ++r) {
        ok[r] = load_box(p, pyr, b, base + (long long)r * blockDim.x, n_b, bx[r], s_lim);
        ba[r] = ok[r] ? area_plus1(bx[r]) : 0.0f;
        best[r] = 0.0f; veq[r] = 0.0f; arg[r] = 0; eq[r] = -1;
    }
    for (int j0 = 0; j0 < K; j0 += kGtChunk) {
        const int kc = min(kGtChunk, K - j0);
        __syncthreads();
        for (int j = threadIdx.x; j < kc; j += blockDim.x) {
            Box t{g[j0 + j], g[p.gt_ld + j0 + j], g[2 * p.gt_ld + j0 + j], g[3 * p.gt_ld + j0 + j]};
            s_gt[j] = t; s_ga[j] = area_plus1(t);
            s_cm[j] = key2f(colmax[(long long)b * p.gt_ld + j0 + j]);
        }
        __syncthreads();
        for (int j = 0; j < kc; ++j) {
            const Box t = s_gt[j];
            const float ta = s_ga[j], cm = s_cm[j];
            const bool cm_ok = cm >= p.min_pos_iou;
            // a miss is +-0: it can only matter as the initial arg-max (GT 0) or when this GT's
            // column max is itself 0 and qualifies (min_pos_iou <= 0) -- both warp-uniform
            const bool need_all = (j0 + j) == 0 || (cm_ok && cm == 0.0f) || !(ta > 0.0f);
#pragma unroll
            for (int r = 0; r < kBoxesPerThread; ++r) {
                if (!ok[r]) continue;
                const bool hit = fmaxf(bx[r].x1, t.x1) < fminf(bx[r].x2, t.x2) && fmaxf(bx[r].y1, t.y1) < fminf(bx[r].y2, t.y2);
                if (!(hit || need_all || !(ba[r] > 0.0f))) continue;
                const float v = iou_plus1(bx[r], ba[r], t, ta);
                if ((j0 + j) == 0 || v > best[r]) { best[r] = v; arg[r] = j0 + j; }       // first max wins
                if (eq[r] < 0 && cm_ok && v == cm) { eq[r] = j0 + j; veq[r] = v; }        // lowest GT wins
            }
        }
    }
    int64_t* lab = labels + (long long)b * p.out_ld;
    float* oiou = out_iou + (long long)b * p.out_ld;
    int* plist = pos_list ? pos_list + (long long)b * pos_cap : nullptr;
#pragma unroll
    for (int r = 0; r < kBoxesPerThread; ++r) {
        const long long i = base + (long long)r * blockDim.x;
        int64_t out_l = -1;
        float out_v = 0.0f;
        const bool in_range = i < n_b;
        if (ok[r]) {
            int l = -1;
            if (best[r] < p.neg_iou) l = 0;
            if (best[r] >= p.pos_iou) l = 1;
            int a = arg[r];
            out_v = best[r];
            if (eq[r] >= 0) { l = 1; a = eq[r]; out_v = veq[r]; }
            out_l = (l == 1) ? (int64_t)(a + 1) : (int64_t)l;
        }
        if (in_range) { lab[lead + i] = out_l; oiou[lead + i] = out_v; }
        const bool is_pos = in_range && out_l > 0, is_neg = in_range && out_l == 0;
        const unsigned mp = __ballot_sync(0xffffffffu, is_pos), mn = __ballot_sync(0xffffffffu, is_neg);
        if (lane_id() == 0) {
            if (mp) atomicAdd(&s_cnt[0], __popc(mp));
            if (mn) atomicAdd(&s_cnt[1], __popc(mn));
        }
        if (plist) {
            const int slot = warp_alloc(is_pos, &census[4 * b + 2]);
            if (is_pos && slot < pos_cap) plist[slot] = (int)(lead + i);
        }
    }
    // prepended GT rows (lib/bbox.py:27-29): labels 1..K, IoU 1
    if (p.prepend_gt && blockIdx.x == 0) {
        for (int j = threadIdx.x; j < K; j += blockDim.x) {
            lab[j] = j + 1; oiou[j] = 1.0f;
            if (plist) { const int slot = atomicAdd(&census[4 * b + 2], 1); if (slot < pos_cap) plist[slot] = j; }
        }
        if (threadIdx.x == 0) atomicAdd(&s_cnt[0], K);
    }
    __syncthreads();
    if (threadIdx.x < 2 && s_cnt[threadIdx.x]) atomicAdd(&census[4 * b + threadIdx.x], s_cnt[threadIdx.x]);
}


// ================= pyramid mode, structure-aware (K2 for anchor heads) ============================
// Anchors are a closed form of (level, a, y, x), so the 94 % of (anchor, GT) pairs that cannot
// intersect never have to be enumerated:
//   k_colmax_rect   CTAs per (GT, level, a, row chunk, image): walk only the cell rectangle whose
//                   anchors can intersect the GT and reduce the exact IoU maximum there (one
//                   atomicMax per CTA).  A GT that no valid anchor intersects keeps "none";
//                   k_label_rows reads that as +0 for valid anchors (a miss is +-0).
//   k_label_rows    a thread owns 4 x-consecutive anchors of one (level, a, y) row -- one index
//                   decomposition per thread instead of one per anchor --, rejects a GT for all 4
//                   with two compares on the row's y-extent, and evaluates the IoU (one IEEE
//                   divide) only for true hits.  128-bit label / IoU stores.
// Both reproduce lib/region.py:75-107 exactly, including the signed zero of max_gt_iou (GT 0 is
// always evaluated in full: it is the first arg-max when nothing overlaps).
constexpr int kRowAnchors = 4;

__device__ __forceinline__ bool anchor_valid(const AssignArgs& p, const Box& a, int y, int x, int in_h, int in_w,
                                             float img_h, float img_w) {
    bool ok = (y < in_h) && (x < in_w);
    if (p.border >= 0.0f)
        ok = ok && a.x1 >= -p.border && a.y1 >= -p.border && a.x2 < img_w + p.border && a.y2 < img_h + p.border;
    return ok;
}

constexpr int kRectChunks = 4;                        // row-interleaved CTAs per (GT, level, a) rectangle

// grid.x enumerates (GT j, level l, anchor a, row chunk rc); colmax holds monotone keys, 0 = "none yet"
__global__ void __launch_bounds__(256) k_colmax_rect(AssignArgs p, b2d_pyramid pyr, uint32_t* __restrict__ colmax,
                                                     int max_a) {
    __shared__ uint32_t s_red[8];
    const int b = blockIdx.y;
    int w = blockIdx.x;
    const int rc = w % kRectChunks; w /= kRectChunks;
    const int a = w % max_a; w /= max_a;
    const int l = w % pyr.num_levels;
    const int j = w / pyr.num_levels;
    if (j >= p.gt_count[b]) return;
    const b2d_level& lv = pyr.lv[l];
    if (a >= lv.A) return;
    const float* g = p.gt + (long long)b * 4 * p.gt_ld;
    const Box t{g[j], g[p.gt_ld + j], g[2 * p.gt_ld + j], g[3 * p.gt_ld + j]};
    const float ta = area_plus1(t);
    const float img_h = p.img_hw[2 * b], img_w = p.img_hw[2 * b + 1];
    int in_h, in_w;
    grid_limits(lv, img_h, img_w, in_h, in_w);
    const float s = lv.stride;
    // cells whose anchor can satisfy max(x1) < min(x2): centre in (g.x1 - w/2, g.x2 + w/2), widened by
    // one cell on each side against rounding; the exact test is iou_plus1's.  A degenerate GT (area
    // not > 0: even a miss may be NaN / inf) scans the whole level.
    const float hw = lv.ws[a] / 2.0f, hh = lv.hs[a] / 2.0f, off = lv.center_lt ? 0.0f : s / 2.0f;
    int x0 = 0, x1 = lv.W - 1, y0 = 0, y1 = lv.H - 1;
    if (ta > 0.0f) {
        x0 = max(0, (int)floorf((t.x1 - hw - off) / s) - 1);
        x1 = min(lv.W - 1, (int)ceilf((t.x2 + hw - off) / s) + 1);
        y0 = max(0, (int)floorf((t.y1 - hh - off) / s) - 1);
        y1 = min(lv.H - 1, (int)ceilf((t.y2 + hh - off) / s) + 1);
    }
    const int rw = x1 - x0 + 1;
    uint32_t m = 0u;
    if (rw > 0) {
        // thread -> (row within my chunk, x): rows y0 + rc, y0 + rc + kRectChunks, ...
        const int tx = threadIdx.x % 64, ty = threadIdx.x / 64;           // 64 x 4 tile of the rectangle
        for (int y = y0 + rc + ty * kRectChunks; y <= y1; y += 4 * kRectChunks) {
            for (int x = x0 + tx; x <= x1; x += 64) {
                const Box an = anchor_at(lv, a, y, x);
                if (!anchor_valid(p, an, y, x, in_h, in_w, img_h, img_w)) continue;
                m = max(m, f2key(iou_plus1(an, area_plus1(an), t, ta) + 0.0f));   // -0 -> +0
            }
        }
    }
    m = __reduce_max_sync(0xffffffffu, m);
    if (lane_id() == 0) s_red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int q = 1; q < 8; ++q) m = max(m, s_red[q]);
        if (m) atomicMax(&colmax[(long long)b * p.gt_ld + j], m);
    }
}

__global__ void __launch_bounds__(256) k_label_rows(AssignArgs p, b2d_pyramid pyr, const uint32_t* __restrict__ colmax,
                                                    int64_t* __restrict__ labels, float* __restrict__ out_iou,
                                                    int* __restrict__ census, int* __restrict__ pos_list, int pos_cap) {
    __shared__ Box s_gt[kGtChunk];
    __shared__ float s_ga[kGtChunk];
    __shared__ float s_cm[kGtChunk];
    __shared__ unsigned char s_all[kGtChunk];        // GT must be evaluated for every anchor (see below)
    __shared__ int s_cnt[2];
    const int b = blockIdx.y;
    const int K = p.gt_count[b];
    const float* g = p.gt + (long long)b * 4 * p.gt_ld;
    const float img_h = p.img_hw[2 * b], img_w = p.img_hw[2 * b + 1];
    if (threadIdx.x < 2) s_cnt[threadIdx.x] = 0;
    // ---- my 4 anchors: flattened index i0 .. i0+3 of the level-major concatenation
    const long long i0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * kRowAnchors;
    Box bx[kRowAnchors];
    float ba[kRowAnchors], best[kRowAnchors], veq[kRowAnchors];
    int arg[kRowAnchors], eq[kRowAnchors];
    bool ok[kRowAnchors], live[kRowAnchors];
    float ylo = INFINITY, yhi = -INFINITY;            // y-extent of my valid anchors (they share a row, mostly)
    {
        int l = -1, a = 0, y = 0, x = 0, in_h = 0, in_w = 0;
        long long lend = -1;                          // first flattened index past the current level
#pragma unroll
        for (int q = 0; q < kRowAnchors; ++q) {
            const long long i = i0 + q;
            live[q] = i < pyr.total;
            ok[q] = false;
            bx[q] = Box{0.f, 0.f, 0.f, 0.f};
            if (live[q]) {
                if (i >= lend) {                      // first element, or the group crosses a level end
                    l = 0;
                    for (int r = 1; r < pyr.num_levels; ++r) if (i >= pyr.lv[r].offset) l = r;
                    const b2d_level& nv = pyr.lv[l];
                    const int li = (int)(i - nv.offset), hw = nv.H * nv.W;
                    a = li / hw;
                    const int r2 = li - a * hw;
                    y = r2 / nv.W; x = r2 - y * nv.W;
                    lend = nv.offset + (long long)nv.A * hw;
                    grid_limits(nv, img_h, img_w, in_h, in_w);
                }
                const b2d_level& lv = pyr.lv[l];
                bx[q] = anchor_at(lv, a, y, x);
                ok[q] = anchor_valid(p, bx[q], y, x, in_h, in_w, img_h, img_w);
                if (++x == lv.W) { x = 0; if (++y == lv.H) { y = 0; ++a; } }
            }
            ba[q] = ok[q] ? area_plus1(bx[q]) : 0.0f;
            if (ok[q]) { ylo = fminf(ylo, bx[q].y1); yhi = fmaxf(yhi, bx[q].y2); }
            best[q] = 0.0f; veq[q] = 0.0f; arg[q] = 0; eq[q] = -1;
        }
    }
    for (int j0 = 0; j0 < K; j0 += kGtChunk) {
        const int kc = min(kGtChunk, K - j0);
        __syncthreads();
        for (int j = threadIdx.x; j < kc; j += blockDim.x) {
            Box t{g[j0 + j], g[p.gt_ld + j0 + j], g[2 * p.gt_ld + j0 + j], g[3 * p.gt_ld + j0 + j]};
            const float ta = area_plus1(t);
            // column max over VALID anchors; an anchor that exists contributes at least a +-0
            const uint32_t ck = colmax[(long long)b * p.gt_ld + j0 + j];
            const float cm = ck ? fmaxf(key2f(ck), 0.0f) : 0.0f;
            s_gt[j] = t; s_ga[j] = ta; s_cm[j] = cm;
            // a miss is +-0: it only matters as the initial arg-max (GT 0), when this GT's column max is
            // itself 0 and qualifies (min_pos_iou <= 0), or when the GT is degenerate (IoU may be NaN)
            s_all[j] = ((j0 + j) == 0 || (cm >= p.min_pos_iou && cm == 0.0f) || !(ta > 0.0f)) ? 1 : 0;
        }
        __syncthreads();
        for (int j = 0; j < kc; ++j) {
            const Box t = s_gt[j];
            const bool all = s_all[j] != 0;
            if (!all && !(fmaxf(ylo, t.y1) < fminf(yhi, t.y2))) continue;      // no valid anchor of mine overlaps in y
            const float ta = s_ga[j], cm = s_cm[j];
            const bool cm_ok = cm >= p.min_pos_iou;
#pragma unroll
            for (int q = 0; q < kRowAnchors; ++q) {
                if (!ok[q]) continue;
                const bool hit = fmaxf(bx[q].x1, t.x1) < fminf(bx[q].x2, t.x2) && fmaxf(bx[q].y1, t.y1) < fminf(bx[q].y2, t.y2);
                if (!(hit || all || !(ba[q] > 0.0f))) continue;
                const float v = iou_plus1(bx[q], ba[q], t, ta);
                if ((j0 + j) == 0 || v > best[q]) { best[q] = v; arg[q] = j0 + j; }       // first max wins
                if (eq[q] < 0 && cm_ok && v == cm) { eq[q] = j0 + j; veq[q] = v; }        // lowest GT wins
            }
        }
    }
    int64_t* lab = labels + (long long)b * p.out_ld;
    float* oiou = out_iou + (long long)b * p.out_ld;
    int* plist = pos_list ? pos_list + (long long)b * pos_cap : nullptr;
    int64_t ol[kRowAnchors];
    float ov[kRowAnchors];
#pragma unroll
    for (int q = 0; q < kRowAnchors; ++q) {
        ol[q] = -1; ov[q] = 0.0f;
        if (ok[q]) {
            int lb = -1;
            if (best[q] < p.neg_iou) lb = 0;
            if (best[q] >= p.pos_iou) lb = 1;
            int a = arg[q];
            ov[q] = best[q];
            if (eq[q] >= 0) { lb = 1; a = eq[q]; ov[q] = veq[q]; }
            ol[q] = (lb == 1) ? (int64_t)(a + 1) : (int64_t)lb;
        }
    }
    const bool vec = live[kRowAnchors - 1] && ((reinterpret_cast<uintptr_t>(lab) & 15) == 0) &&
                     ((reinterpret_cast<uintptr_t>(oiou) & 15) == 0);     // i0 is a multiple of 4
    if (vec) {
        reinterpret_cast<longlong2*>(lab + i0)[0] = make_longlong2(ol[0], ol[1]);
        reinterpret_cast<longlong2*>(lab + i0)[1] = make_longlong2(ol[2], ol[3]);
        *reinterpret_cast<float4*>(oiou + i0) = make_float4(ov[0], ov[1], ov[2], ov[3]);
    } else {
#pragma unroll
        for (int q = 0; q < kRowAnchors; ++q)
            if (live[q]) { lab[i0 + q] = ol[q]; oiou[i0 + q] = ov[q]; }
    }
#pragma unroll
    for (int q = 0; q < kRowAnchors; ++q) {
        const bool is_pos = live[q] && ol[q] > 0, is_neg = live[q] && ol[q] == 0;
        const unsigned mp = __ballot_sync(0xffffffffu, is_pos), mn = __ballot_sync(0xffffffffu, is_neg);
        if (lane_id() == 0) {
            if (mp) atomicAdd(&s_cnt[0], __popc(mp));
            if (mn) atomicAdd(&s_cnt[1], __popc(mn));
        }
        if (plist) {
            const int slot = warp_alloc(is_pos, &census[4 * b + 2]);
            if (is_pos && slot < pos_cap) plist[slot] = (int)(i0 + q);
        }
    }
    __syncthreads();
    if (threadIdx.x < 2 && s_cnt[threadIdx.x]) atomicAdd(&census[4 * b + threadIdx.x], s_cnt[threadIdx.x]);
}

// ---- small problems (explicit boxes, N <= 4096: the RoI-target assignment of 2000 proposals) ----
// colmax + label + census in ONE launch, one CTA per image: the two-pass grid version costs two
// launches of 16 CTAs whose time is pure launch + global-atomic latency (14 + 14 us, ncu r1e).
// s_lab (optional, shared memory, >= lead + n_b entries): the labels as int32, for the fused kernel below
__device__ __forceinline__ void assign_small_body(const AssignArgs& p, SmallSmem& sm, int64_t* __restrict__ labels,
                                                  float* __restrict__ out_iou, int* __restrict__ census,
                                                  int* __restrict__ pos_list, int pos_cap, int* s_lab) {
    Box* s_gt = sm.gt;
    float* s_ga = sm.ga;
    uint32_t* s_max = sm.mx;
    int* s_cnt = sm.cnt;
    const int b = blockIdx.x;
    const int K = p.gt_count[b];
    const int n_b = p.box_count ? p.box_count[b] : (int)p.N;
    const float* g = p.gt + (long long)b * 4 * p.gt_ld;
    const float* src = p.boxes + (long long)b * 4 * p.box_ld;
    const int lead = p.prepend_gt ? K : 0;
    const uint32_t kNegInf = f2key(-INFINITY);
    if (threadIdx.x < 3) s_cnt[threadIdx.x] = 0;
    for (int j = threadIdx.x; j < K; j += blockDim.x) {
        Box t{g[j], g[p.gt_ld + j], g[2 * p.gt_ld + j], g[3 * p.gt_ld + j]};
        s_gt[j] = t; s_ga[j] = area_plus1(t); s_max[j] = kNegInf;
    }
    Box bx[kSmallBoxes];
    float ba[kSmallBoxes];
    bool ok[kSmallBoxes];
#pragma unroll
    for (int r = 0; r < kSmallBoxes; ++r) {
        const int i = threadIdx.x + r * kSmallThreads;
        ok[r] = i < n_b;
        if (ok[r]) bx[r] = Box{src[i], src[p.box_ld + i], src[2 * p.box_ld + i], src[3 * p.box_ld + i]};
        else bx[r] = Box{0.f, 0.f, 0.f, 0.f};
        ba[r] = ok[r] ? area_plus1(bx[r]) : 0.0f;
    }
    __syncthreads();
    // pass 1: per-GT column max (lib/region.py:86), -0 folded to +0 like the grid kernel
    for (int j = 0; j < K; ++j) {
        const Box t = s_gt[j];
        const float ta = s_ga[j];
        uint32_t m = kNegInf;
#pragma unroll
        for (int r = 0; r < kSmallBoxes; ++r)
            if (ok[r]) m = max(m, f2key(iou_plus1(bx[r], ba[r], t, ta) + 0.0f));
        m = __reduce_max_sync(0xffffffffu, m);
        if (lane_id() == 0 && m != kNegInf) atomicMax(&s_max[j], m);
    }
    __syncthreads();
    // pass 2: labels (lib/region.py:88-107)
    float best[kSmallBoxes], veq[kSmallBoxes];
    int arg[kSmallBoxes], eq[kSmallBoxes];
#pragma unroll
    for (int r = 0; r < kSmallBoxes; ++r) { best[r] = 0.0f; veq[r] = 0.0f; arg[r] = 0; eq[r] = -1; }
    for (int j = 0; j < K; ++j) {
        const Box t = s_gt[j];
        const float ta = s_ga[j], cm = key2f(s_max[j]);
        const bool cm_ok = cm >= p.min_pos_iou;
#pragma unroll
        for (int r = 0; r < kSmallBoxes; ++r) {
            if (!ok[r]) continue;
            const float v = iou_plus1(bx[r], ba[r], t, ta);
            if (j == 0 || v > best[r]) { best[r] = v; arg[r] = j; }            // first max wins
            if (eq[r] < 0 && cm_ok && v == cm) { eq[r] = j; veq[r] = v; }      // lowest GT wins
        }
    }
    int64_t* lab = labels + (long long)b * p.out_ld;
    float* oiou = out_iou + (long long)b * p.out_ld;
    int* plist = pos_list ? pos_list + (long long)b * pos_cap : nullptr;
#pragma unroll
    for (int r = 0; r < kSmallBoxes; ++r) {
        const int i = threadIdx.x + r * kSmallThreads;
        int64_t out_l = -1;
        float out_v = 0.0f;
        if (ok[r]) {
            int l = -1;
            if (best[r] < p.neg_iou) l = 0;
            if (best[r] >= p.pos_iou) l = 1;
            int a = arg[r];
            out_v = best[r];
            if (eq[r] >= 0) { l = 1; a = eq[r]; out_v = veq[r]; }
            out_l = (l == 1) ? (int64_t)(a + 1) : (int64_t)l;
            lab[lead + i] = out_l; oiou[lead + i] = out_v;
            if (s_lab) s_lab[lead + i] = (int)out_l;
        }
        const bool is_pos = ok[r] && out_l > 0, is_neg = ok[r] && out_l == 0;
        const unsigned mp = __ballot_sync(0xffffffffu, is_pos), mn = __ballot_sync(0xffffffffu, is_neg);
        if (lane_id() == 0) {
            if (mp) atomicAdd(&s_cnt[0], __popc(mp));
            if (mn) atomicAdd(&s_cnt[1], __popc(mn));
        }
        if (plist) {
            const int slot = warp_alloc(is_pos, &s_cnt[2]);
            if (is_pos && slot < pos_cap) plist[slot] = lead + i;
        }
    }
    __syncthreads();
    if (p.prepend_gt) {                                   // prepended GT rows (lib/bbox.py:27-29): labels 1..K, IoU 1
        for (int j = threadIdx.x; j < K; j += blockDim.x) {
            lab[j] = j + 1; oiou[j] = 1.0f;
            if (s_lab) s_lab[j] = j + 1;
            if (plist) { const int slot = atomicAdd(&s_cnt[2], 1); if (slot < pos_cap) plist[slot] = j; }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        census[4 * b + 0] = s_cnt[0] + (p.prepend_gt ? K : 0);
        census[4 * b + 1] = s_cnt[1];
        census[4 * b + 2] = s_cnt[2];
        census[4 * b + 3] = 0;
    }
    __syncthreads();
}

__global__ void __launch_bounds__(kSmallThreads) k_assign_small(AssignArgs p, int64_t* __restrict__ labels,
                                                                float* __restrict__ out_iou, int* __restrict__ census,
                                                                int* __restrict__ pos_list, int pos_cap) {
    __shared__ SmallSmem sm;
    assign_small_body(p, sm, labels, out_iou, census, pos_list, pos_cap, nullptr);
}

// ---- census of an arbitrary labels vector -------------------------------------
__global__ void __launch_bounds__(256) k_label_census(int* __restrict__ census, int* __restrict__ pos_list,
                                                      int pos_cap, const int64_t* __restrict__ labels,
                                                      long long ld, const int* __restrict__ count, long long n) {
    __shared__ int s_cnt[2];
    const int b = blockIdx.y;
    if (threadIdx.x < 2) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    const long long n_b = count ? (long long)count[b] : n;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t l = (i < n_b) ? labels[(long long)b * ld + i] : -1;
    const bool is_pos = l > 0, is_neg = (i < n_b) && l == 0;
    const unsigned mp = __ballot_sync(0xffffffffu, is_pos), mn = __ballot_sync(0xffffffffu, is_neg);
    if (lane_id() == 0) {
        if (mp) atomicAdd(&s_cnt[0], __popc(mp));
        if (mn) atomicAdd(&s_cnt[1], __popc(mn));
    }
    if (pos_list) {
        const int slot = warp_alloc(is_pos, &census[4 * b + 2]);
        if (is_pos && slot < pos_cap) pos_list[(long long)b * pos_cap + slot] = (int)i;
    }
    __syncthreads();
    if (threadIdx.x < 2 && s_cnt[threadIdx.x]) atomicAdd(&census[4 * b + threadIdx.x], s_cnt[threadIdx.x]);
}

// ---- device-RNG sampler (spec: DESIGN.md "Samplers"; oracle/sampler_spec.py) ----
// positives: if #pos > pos_num keep the pos_num smallest (mix_key(seed, idx), idx).
// negatives: walk the keyed Feistel permutation of [0, n) and keep the first
// (max_num - #kept_pos) indices whose label is 0.  Output ascending.
constexpr int kSampleThreads = 1024;
constexpr int kSampleSortCap = 4096;

__global__ void __launch_bounds__(kSampleThreads) k_sample(int* __restrict__ chosen, int* __restrict__ n_chosen,
                                                           const int64_t* __restrict__ labels, long long ld,
                                                           const int* __restrict__ count,
                                                           const int* __restrict__ count_add, long long n,
                                                           const int* __restrict__ census,
                                                           const int* __restrict__ pos_list, int pos_cap,
                                                           int max_num, int pos_num, unsigned long long seed,
                                                           const unsigned long long* __restrict__ seed_step) {
    extern __shared__ __align__(16) uint64_t s_sort[];          // kSampleSortCap entries
    if (seed_step) seed += *seed_step;                            // per-step counter in device memory (CUDA-graph replays)
    __shared__ int s_n, s_warp[kSampleThreads / 32], s_take;
    __shared__ unsigned long long s_lo, s_hi;
    const int b = blockIdx.x;
    const int64_t* lab = labels + (long long)b * ld;
    const long long n_b = (count ? (long long)count[b] : n) + (count_add ? (long long)count_add[b] : 0);
    const int npos = min(census[4 * b + 0], pos_cap);
    const int nneg = census[4 * b + 1];
    const int* plist = pos_list + (long long)b * pos_cap;
    const uint64_t sd = seed + 0x632BE59BD9B4E019ull * (uint64_t)(b + 1);
    int* out = chosen + (long long)b * max_num;
    if (threadIdx.x == 0) s_n = 0;
    __syncthreads();

    // ---- positives
    const int keep_pos = min(npos, pos_num);
    uint64_t thr = ~0ull;   // keep composites <= thr
    if (npos > pos_num) {
        // 64-step bisection for the pos_num-th smallest composite (key<<32 | idx): exact, order-free
        if (threadIdx.x == 0) { s_lo = 0ull; s_hi = ~0ull; }
        __syncthreads();
        for (int it = 0; it < 64; ++it) {
            const unsigned long long lo = s_lo, hi = s_hi;
            if (lo >= hi) break;
            const unsigned long long mid = lo + (hi - lo) / 2;
            int c = 0;
            for (int t = threadIdx.x; t < npos; t += blockDim.x) {
                const uint32_t idx = (uint32_t)plist[t];
                const uint64_t comp = ((uint64_t)mix_key(sd, idx) << 32) | idx;
                c += (comp <= mid);
            }
            c = __reduce_add_sync(0xffffffffu, c);
            if (lane_id() == 0) s_warp[threadIdx.x >> 5] = c;
            __syncthreads();
            if (threadIdx.x == 0) {
                int tot = 0;
                for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += s_warp[w];
                if (tot >= pos_num) s_hi = mid; else s_lo = mid + 1;
            }
            __syncthreads();
        }
        thr = s_lo;
    }
    for (int t0 = 0; t0 < npos; t0 += blockDim.x) {
        const int t = t0 + threadIdx.x;
        bool take = false;
        uint32_t idx = 0;
        if (t < npos) {
            idx = (uint32_t)plist[t];
            take = (((uint64_t)mix_key(sd, idx) << 32) | idx) <= thr;
        }
        const int slot = warp_alloc(take, &s_n);
        if (take && slot < kSampleSortCap) s_sort[slot] = (uint64_t)idx;
    }
    __syncthreads();
    // ---- negatives
    const int want_neg = min(max(max_num - keep_pos, 0), nneg);
    if (want_neg > 0) {
        int bits = 2;
        while ((1ll << bits) < n_b) ++bits;
        if (bits & 1) ++bits;
        const int half = bits >> 1;
        const long long dom = 1ll << bits;
        if (threadIdx.x == 0) s_take = 0;
        __syncthreads();
        if (blockDim.x <= 256) {
            // slim launch (128 threads: a CTA that fits the hole one retiring RoIAlign CTA leaves, see fused.TrainHotPath):
            // 4 permutation steps per thread and round, so that 4 label loads are in flight per thread; same order by t
            __shared__ int s_cnt4[4][8];
            const int nw = blockDim.x >> 5, wq = threadIdx.x >> 5;
            for (long long t0 = 0; t0 < dom; t0 += 4ll * blockDim.x) {
                uint32_t y[4];
                bool hit[4];
                unsigned m[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const long long t = t0 + (long long)q * blockDim.x + threadIdx.x;
                    y[q] = feistel((uint32_t)t, half, sd ^ 0xA5A5A5A5DEADBEEFull);
                    hit[q] = t < dom && ((long long)y[q] < n_b) && (lab[y[q]] == 0);
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    m[q] = __ballot_sync(0xffffffffu, hit[q]);
                    if (lane_id() == 0) s_cnt4[q][wq] = __popc(m[q]);
                }
                __syncthreads();
                int before = s_take, tot = 0;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    int mine = before + tot;
                    for (int w = 0; w < nw; ++w) { if (w < wq) mine += s_cnt4[q][w]; tot += s_cnt4[q][w]; }
                    const int rank = mine + __popc(m[q] & ((1u << lane_id()) - 1u));
                    if (hit[q] && rank < want_neg) s_sort[keep_pos + rank] = (uint64_t)y[q];
                }
                __syncthreads();
                if (threadIdx.x == 0) s_take += tot;
                __syncthreads();
                if (s_take >= want_neg) break;
            }
        } else
        for (long long t0 = 0; t0 < dom; t0 += blockDim.x) {
            const uint32_t y = feistel((uint32_t)(t0 + threadIdx.x), half, sd ^ 0xA5A5A5A5DEADBEEFull);
            const bool hit = ((long long)y < n_b) && (lab[y] == 0);
            // ordered (by t) slot assignment: block-wide exclusive scan of hits
            const unsigned m = __ballot_sync(0xffffffffu, hit);
            if (lane_id() == 0) s_warp[threadIdx.x >> 5] = __popc(m);
            __syncthreads();
            int before = s_take;
            for (int w = 0; w < (threadIdx.x >> 5); ++w) before += s_warp[w];
            const int rank = before + __popc(m & ((1u << lane_id()) - 1u));
            if (hit && rank < want_neg) s_sort[keep_pos + rank] = (uint64_t)y;
            __syncthreads();
            if (threadIdx.x == 0) {
                int tot = 0;
                for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += s_warp[w];
                s_take += tot;
            }
            __syncthreads();
            if (s_take >= want_neg) break;
        }
    }
    __syncthreads();
    const int total = keep_pos + want_neg;
    int p2 = 1;
    while (p2 < total) p2 <<= 1;
    // ascending index == descending (~idx); pad with 0 (sorts last)
    for (int t = threadIdx.x; t < p2; t += blockDim.x)
        s_sort[t] = (t < total) ? (0xffffffffull - s_sort[t]) + 1ull : 0ull;
    __syncthreads();
    bitonic_sort_desc(s_sort, p2);
    for (int t = threadIdx.x; t < max_num; t += blockDim.x)
        out[t] = (t < total) ? (int)(0xffffffffull - (s_sort[t] - 1ull)) : -1;
    if (threadIdx.x == 0) n_chosen[b] = total;
}

__global__ void __launch_bounds__(256) k_scatter_sampled(int64_t* __restrict__ out, const int64_t* __restrict__ labels,
                                                         long long ld, const int* __restrict__ chosen,
                                                         const int* __restrict__ n_chosen, int max_num) {
    const int b = blockIdx.y;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_chosen[b]) return;
    const int i = chosen[(long long)b * max_num + t];
    out[(long long)b * ld + i] = labels[(long long)b * ld + i];
}

// ---- fused gather + encode of the sampled rows ---------------------------------
struct EncArgs {
    const int* chosen; const int* n_chosen; int max_num;
    const int64_t* labels; long long label_ld;
    const float* boxes; long long box_ld; int use_pyr;
    const float* gt; int gt_ld; const int* gt_count; const int64_t* gt_label;
    int prepend_gt;
    float ms[8];
};

__global__ void __launch_bounds__(128) k_encode_targets(EncArgs p, b2d_pyramid pyr, float* __restrict__ tar_box,
                                                        float* __restrict__ tar_gt, float* __restrict__ tar_param,
                                                        int64_t* __restrict__ tar_label,
                                                        int64_t* __restrict__ tar_is_gt) {
    const int b = blockIdx.y;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= p.max_num) return;
    const long long o = (long long)b * 4 * p.max_num;
    const bool live = t < p.n_chosen[b];
    Box bx{0, 0, 0, 0}, gb{0, 0, 0, 0};
    float prm[4] = {0, 0, 0, 0};
    int64_t lab_out = 0, isgt = 0;
    if (live) {
        const int K = p.gt_count[b];
        const int lead = p.prepend_gt ? K : 0;
        const int i = p.chosen[(long long)b * p.max_num + t];
        const int64_t lab = p.labels[(long long)b * p.label_ld + i];
        const float* g = p.gt + (long long)b * 4 * p.gt_ld;
        if (i < lead) {
            bx = Box{g[i], g[p.gt_ld + i], g[2 * p.gt_ld + i], g[3 * p.gt_ld + i]};
            isgt = 1;
        } else if (p.use_pyr) {
            const long long ii = i - lead;
            int l = 0;
            for (int q = 1; q < pyr.num_levels; ++q)
                if (ii >= pyr.lv[q].offset) l = q;
            bx = anchor_flat(pyr.lv[l], (int)(ii - pyr.lv[l].offset));
        } else {
            const float* src = p.boxes + (long long)b * 4 * p.box_ld;
            const long long ii = i - lead;
            bx = Box{src[ii], src[p.box_ld + ii], src[2 * p.box_ld + ii], src[3 * p.box_ld + ii]};
        }
        const int j = (int)max(lab - 1, (int64_t)0);        // negatives point at GT 0 (lib/anchor.py:45-47)
        gb = Box{g[j], g[p.gt_ld + j], g[2 * p.gt_ld + j], g[3 * p.gt_ld + j]};
        const float bw = (bx.x2 - bx.x1) + 1.0f, bh = (bx.y2 - bx.y1) + 1.0f;
        const float gw = (gb.x2 - gb.x1) + 1.0f, gh = (gb.y2 - gb.y1) + 1.0f;
        const float bcx = (bx.x2 + bx.x1) / 2.0f, bcy = (bx.y2 + bx.y1) / 2.0f;
        const float gcx = (gb.x2 + gb.x1) / 2.0f, gcy = (gb.y2 + gb.y1) / 2.0f;
        prm[0] = ((gcx - bcx) / bw - p.ms[0]) / p.ms[4];
        prm[1] = ((gcy - bcy) / bh - p.ms[1]) / p.ms[5];
        prm[2] = (logf(gw / bw) - p.ms[2]) / p.ms[6];
        prm[3] = (logf(gh / bh) - p.ms[3]) / p.ms[7];
        if (p.gt_label) lab_out = (lab > 0) ? p.gt_label[(long long)b * p.gt_ld + j] : 0;
        else lab_out = (lab > 0) ? 1 : 0;
    }
    if (tar_box) { tar_box[o + t] = bx.x1; tar_box[o + p.max_num + t] = bx.y1; tar_box[o + 2 * p.max_num + t] = bx.x2; tar_box[o + 3 * p.max_num + t] = bx.y2; }
    if (tar_gt) { tar_gt[o + t] = gb.x1; tar_gt[o + p.max_num + t] = gb.y1; tar_gt[o + 2 * p.max_num + t] = gb.x2; tar_gt[o + 3 * p.max_num + t] = gb.y2; }
    if (tar_param) { tar_param[o + t] = prm[0]; tar_param[o + p.max_num + t] = prm[1]; tar_param[o + 2 * p.max_num + t] = prm[2]; tar_param[o + 3 * p.max_num + t] = prm[3]; }
    if (tar_label) tar_label[(long long)b * p.max_num + t] = lab_out;
    if (tar_is_gt) tar_is_gt[(long long)b * p.max_num + t] = isgt;
}

// ---- gather of the head outputs at the sampled anchors (lib/anchor.py:49-56) ----------
struct GatherArgs {
    const float* cls[kMaxLevels]; const float* reg[kMaxLevels];
    const int* chosen; const int* n_chosen; int max_num, cls_ch;
};

__global__ void __launch_bounds__(128) k_gather_head(GatherArgs p, b2d_pyramid pyr, float* __restrict__ tar_cls,
                                                     float* __restrict__ tar_reg) {
    const int b = blockIdx.y;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= p.max_num) return;
    const bool live = t < p.n_chosen[b];
    int l = 0, li = 0;
    long long n = 1;
    if (live) {
        const int i = p.chosen[(long long)b * p.max_num + t];
        for (int q = 1; q < pyr.num_levels; ++q) if (i >= pyr.lv[q].offset) l = q;
        li = (int)(i - pyr.lv[l].offset);
        n = (long long)pyr.lv[l].A * pyr.lv[l].H * pyr.lv[l].W;
    }
    for (int c = 0; c < p.cls_ch; ++c)
        tar_cls[((long long)b * p.cls_ch + c) * p.max_num + t] = live ? p.cls[l][((long long)b * p.cls_ch + c) * n + li] : 0.0f;
    for (int c = 0; c < 4; ++c)
        tar_reg[((long long)b * 4 + c) * p.max_num + t] = live ? p.reg[l][((long long)b * 4 + c) * n + li] : 0.0f;
}

// ---- adjoint of k_gather_head: the dense head-map gradients from the gradients at the sampled anchors ----------
// A thread owns kScatterRun consecutive elements of one plane (image b, level l, channel: cls_ch class planes, then 4
// regression planes) and writes each of them exactly once: the upstream value where the anchor was sampled, zero
// elsewhere -- no memset, no atomics.  Precondition (DESIGN §8, every sampler of this library): chosen[b][0 .. n_chosen[b])
// is ascending and free of duplicates; its first sample at or after the run is found by binary search.
constexpr int kScatterRun = 16;

struct ScatterArgs {
    float* cls[kMaxLevels]; float* reg[kMaxLevels];
    const float* g_cls; const float* g_reg;
    const int* chosen; const int* n_chosen; int max_num, cls_ch;
    long long run_off[kMaxLevels + 1];     // first run of each level within an image
};

__global__ void __launch_bounds__(256) k_scatter_head(ScatterArgs p, b2d_pyramid pyr) {
    const int b = blockIdx.y;
    long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= p.run_off[pyr.num_levels]) return;
    int l = 0;
    for (int q = 1; q < pyr.num_levels; ++q) if (t >= p.run_off[q]) l = q;
    t -= p.run_off[l];
    const long long n = (long long)pyr.lv[l].A * pyr.lv[l].H * pyr.lv[l].W;
    const long long runs = (n + kScatterRun - 1) / kScatterRun;
    const int plane = (int)(t / runs);
    const long long li0 = (t - plane * runs) * kScatterRun;
    const int len = (int)min((long long)kScatterRun, n - li0);
    float* dst;
    const float* g;
    if (plane < p.cls_ch) {
        dst = p.cls[l] + ((long long)b * p.cls_ch + plane) * n + li0;
        g = p.g_cls + ((long long)b * p.cls_ch + plane) * p.max_num;
    } else {
        dst = p.reg[l] + ((long long)b * 4 + plane - p.cls_ch) * n + li0;
        g = p.g_reg + ((long long)b * 4 + plane - p.cls_ch) * p.max_num;
    }
    const int* ch = p.chosen + (long long)b * p.max_num;
    const int cnt = min(p.n_chosen[b], p.max_num);
    const long long base = pyr.lv[l].offset + li0;          // flat anchor index of the run's first element
    int lo = 0, hi = cnt;                                   // first sample >= base
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if ((long long)__ldg(ch + mid) < base) lo = mid + 1; else hi = mid;
    }
    int j = lo;
    int nxt = j < cnt ? (int)min((long long)__ldg(ch + j) - base, (long long)kScatterRun) : kScatterRun;
    float v[kScatterRun];
#pragma unroll
    for (int e = 0; e < kScatterRun; ++e) {
        float x = 0.0f;
        if (e == nxt) {
            x = __ldg(g + j);
            ++j;
            nxt = j < cnt ? (int)min((long long)__ldg(ch + j) - base, (long long)kScatterRun) : kScatterRun;
        }
        v[e] = x;
    }
    if (len == kScatterRun && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
#pragma unroll
        for (int e = 0; e < kScatterRun; e += 4)
            *reinterpret_cast<float4*>(dst + e) = make_float4(v[e], v[e + 1], v[e + 2], v[e + 3]);
    } else {
#pragma unroll
        for (int e = 0; e < kScatterRun; ++e)
            if (e < len) dst[e] = v[e];
    }
}

// ---- bbox_target of one image in ONE launch (lib/bbox.py:6-82) -----------------------------------
// assignment (assign_small_body) -> device-RNG sampler (the specification of k_sample,
// oracle/sampler_spec.py: identical `chosen`) -> gather + encode (k_encode_targets), one CTA per
// image, labels / flags in shared memory.  Replaces three dependent launches of 8 CTAs (13 + 17 +
// 5 us + gaps on the critical path of config 2); the negative walk is one block scan per 4096
// permutation steps and the ascending output order comes from a flag compaction, not a sort.
__global__ void __launch_bounds__(kSmallThreads) k_roi_targets_small(AssignArgs p, int64_t* __restrict__ labels,
                                                                     float* __restrict__ out_iou,
                                                                     int* __restrict__ census, int* __restrict__ pos_list,
                                                                     int pos_cap, FusedArgs f) {
    __shared__ SmallSmem sm;
    __shared__ FusedScratch fs;
    pdl_wait();                                         // the proposals (no-op unless launched as a programmatic dependent)
    assign_small_body(p, sm, labels, out_iou, census, pos_list, pos_cap, fs.lab);
    fused_sample_encode(p, f, sm.gt, fs, sm.cnt[0], sm.cnt[1], blockIdx.x);
}

__global__ void k_counter_add(unsigned long long* cell, unsigned long long inc) { *cell += inc; }

__global__ void k_fill_u32(uint32_t* p, uint32_t v, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

}  // namespace b2d

using namespace b2d;

extern "C" {

int b2d_assign_max_iou(int64_t* labels, float* max_iou, long long out_ld, const float* boxes, long long box_ld,
                       const int* box_count, long long N, const b2d_pyramid* pyr_host, const float* img_hw,
                       float border, const float* gt, int gt_ld, const int* gt_count, int B, float pos_iou,
                       float neg_iou, float min_pos_iou, int prepend_gt, int* census, int* pos_list, int pos_cap,
                       void* workspace, size_t ws_bytes, void* stream) {
    B2D_REQUIRE(labels && max_iou && gt && gt_count && census, "assign_max_iou: null pointer");
    B2D_REQUIRE(boxes || (pyr_host && img_hw), "assign_max_iou: need boxes or pyramid+img_hw");
    B2D_REQUIRE(B >= 1 && gt_ld >= 1 && N >= 0, "assign_max_iou: bad sizes");
    B2D_REQUIRE(workspace && ws_bytes >= (size_t)B * gt_ld * 4, "assign_max_iou: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    AssignArgs a;
    a.boxes = boxes; a.box_ld = box_ld; a.box_count = box_count; a.N = N;
    a.use_pyr = boxes ? 0 : 1; a.img_hw = img_hw; a.border = border;
    a.gt = gt; a.gt_ld = gt_ld; a.gt_count = gt_count;
    a.pos_iou = pos_iou; a.neg_iou = neg_iou; a.min_pos_iou = min_pos_iou;
    a.prepend_gt = prepend_gt; a.out_ld = out_ld;
    b2d_pyramid pyr;
    memset(&pyr, 0, sizeof(pyr));
    if (a.use_pyr) { pyr = *pyr_host; a.N = pyr.total; }
    if (!a.use_pyr && N <= kSmallThreads * kSmallBoxes && gt_ld <= kGtChunk) {
        k_assign_small<<<B, kSmallThreads, 0, st>>>(a, labels, max_iou, census, pos_list, pos_cap);
        return check_launch("assign_max_iou");
    }
    if (a.use_pyr && !prepend_gt && !knobs().assign_old) {
        uint32_t* cmx = (uint32_t*)workspace;
        cudaMemsetAsync(census, 0, sizeof(int) * 4 * B, st);
        cudaMemsetAsync(cmx, 0, sizeof(uint32_t) * (size_t)B * gt_ld, st);
        int max_a = 1;
        for (int l = 0; l < pyr.num_levels; ++l) max_a = max(max_a, pyr.lv[l].A);
        dim3 g1(gt_ld * pyr.num_levels * max_a * kRectChunks, B);
        k_colmax_rect<<<g1, 256, 0, st>>>(a, pyr, cmx, max_a);
        dim3 g2(cdiv(pyr.total, 256 * kRowAnchors), B);
        k_label_rows<<<g2, 256, 0, st>>>(a, pyr, cmx, labels, max_iou, census, pos_list, pos_cap);
        return check_launch("assign_max_iou");
    }
    uint32_t* colmax = (uint32_t*)workspace;
    const long long nc = (long long)B * gt_ld;
    k_fill_u32<<<cdiv(nc, 256), 256, 0, st>>>(colmax, f2key(-INFINITY), nc);
    cudaMemsetAsync(census, 0, sizeof(int) * 4 * B, st);
    const int per_block = 256 * kBoxesPerThread;
    dim3 grid(cdiv(a.N > 0 ? a.N : 1, per_block), B);
    k_assign_colmax<<<grid, 256, 0, st>>>(a, pyr, colmax);
    k_assign_label<<<grid, 256, 0, st>>>(a, pyr, colmax, labels, max_iou, census, pos_list, pos_cap);
    return check_launch("assign_max_iou");
}

int b2d_label_census(int* census, int* pos_list, int pos_cap, const int64_t* labels, long long ld,
                     const int* count, long long n, int B, void* stream) {
    B2D_REQUIRE(census && labels && B >= 1 && n >= 0, "label_census: bad args");
    cudaStream_t st = (cudaStream_t)stream;
    cudaMemsetAsync(census, 0, sizeof(int) * 4 * B, st);
    if (n == 0) return B2D_OK;
    dim3 grid(cdiv(n, 256), B);
    k_label_census<<<grid, 256, 0, st>>>(census, pos_list, pos_cap, labels, ld, count, n);
    return check_launch("label_census");
}

int b2d_sample_labels(int* chosen, int* n_chosen, const int64_t* labels, long long ld, const int* count,
                      const int* count_add, long long n, const int* census, const int* pos_list, int pos_cap, int B, int max_num,
                      int pos_num, unsigned long long seed, const unsigned long long* seed_step, void* stream) {
    B2D_REQUIRE(chosen && n_chosen && labels && census && pos_list, "sample_labels: null pointer");
    B2D_REQUIRE(B >= 1 && max_num >= 1 && max_num <= kSampleSortCap && pos_num >= 0 && pos_num <= max_num,
                "sample_labels: need 1 <= max_num <= 4096 and pos_num <= max_num");
    B2D_REQUIRE(n < (1ll << 31), "sample_labels: n too large");
    // function attributes are per device: set on every call (a process may drive several GPUs)
    B2D_SMEM(k_sample, kSampleSortCap * 8, "k_sample");
    const int threads = (knobs().sample_threads == 128 || knobs().sample_threads == 256) ? knobs().sample_threads : kSampleThreads;
    k_sample<<<B, threads, kSampleSortCap * 8, (cudaStream_t)stream>>>(
        chosen, n_chosen, labels, ld, count, count_add, n, census, pos_list, pos_cap, max_num, pos_num, seed, seed_step);
    return check_launch("sample_labels");
}

int b2d_counter_add(unsigned long long* cell, unsigned long long inc, void* stream) {
    B2D_REQUIRE(cell, "counter_add: null pointer");
    k_counter_add<<<1, 1, 0, (cudaStream_t)stream>>>(cell, inc);
    return check_launch("counter_add");
}

int b2d_scatter_sampled(int64_t* out, const int64_t* labels, long long ld, long long n, const int* chosen,
                        const int* n_chosen, int max_num, int B, void* stream) {
    B2D_REQUIRE(out && labels && chosen && n_chosen && B >= 1, "scatter_sampled: bad args");
    (void)n;
    dim3 grid(cdiv(max_num, 256), B);
    k_scatter_sampled<<<grid, 256, 0, (cudaStream_t)stream>>>(out, labels, ld, chosen, n_chosen, max_num);
    return check_launch("scatter_sampled");
}

int b2d_gather_head_outputs(float* tar_cls, float* tar_reg, const void* const* cls_ptrs_host,
                            const void* const* reg_ptrs_host, const b2d_pyramid* pyr_host, int cls_channels,
                            const int* chosen, const int* n_chosen, int max_num, int B, void* stream) {
    B2D_REQUIRE(tar_cls && tar_reg && cls_ptrs_host && reg_ptrs_host && pyr_host && chosen && n_chosen,
                "gather_head_outputs: null pointer");
    GatherArgs p;
    memset(&p, 0, sizeof(p));
    for (int l = 0; l < pyr_host->num_levels; ++l) { p.cls[l] = (const float*)cls_ptrs_host[l]; p.reg[l] = (const float*)reg_ptrs_host[l]; }
    p.chosen = chosen; p.n_chosen = n_chosen; p.max_num = max_num; p.cls_ch = cls_channels;
    dim3 grid(cdiv(max_num, 128), B);
    k_gather_head<<<grid, 128, 0, (cudaStream_t)stream>>>(p, *pyr_host, tar_cls, tar_reg);
    return check_launch("gather_head_outputs");
}

int b2d_scatter_head_grads(void* const* dcls_ptrs_host, void* const* dreg_ptrs_host, const float* grad_tar_cls,
                           const float* grad_tar_reg, const b2d_pyramid* pyr_host, int cls_channels, const int* chosen,
                           const int* n_chosen, int max_num, int B, void* stream) {
    B2D_REQUIRE(dcls_ptrs_host && dreg_ptrs_host && grad_tar_cls && grad_tar_reg && pyr_host && chosen && n_chosen,
                "scatter_head_grads: null pointer");
    B2D_REQUIRE(B >= 1 && max_num >= 1 && cls_channels >= 1 && pyr_host->num_levels >= 1 &&
                pyr_host->num_levels <= kMaxLevels, "scatter_head_grads: bad sizes");
    ScatterArgs p;
    memset(&p, 0, sizeof(p));
    long long run = 0;
    for (int l = 0; l < pyr_host->num_levels; ++l) {
        B2D_REQUIRE(dcls_ptrs_host[l] && dreg_ptrs_host[l], "scatter_head_grads: null level pointer");
        p.cls[l] = (float*)dcls_ptrs_host[l]; p.reg[l] = (float*)dreg_ptrs_host[l];
        const b2d_level& v = pyr_host->lv[l];
        p.run_off[l] = run;
        run += (long long)(cls_channels + 4) * cdiv((long long)v.A * v.H * v.W, kScatterRun);
    }
    p.run_off[pyr_host->num_levels] = run;
    p.g_cls = grad_tar_cls; p.g_reg = grad_tar_reg;
    p.chosen = chosen; p.n_chosen = n_chosen; p.max_num = max_num; p.cls_ch = cls_channels;
    if (run == 0) return B2D_OK;
    dim3 grid((unsigned)cdiv(run, 256), (unsigned)B);
    k_scatter_head<<<grid, 256, 0, (cudaStream_t)stream>>>(p, *pyr_host);
    return check_launch("scatter_head_grads");
}

int b2d_encode_targets(float* tar_box, float* tar_gt, float* tar_param, int64_t* tar_label, int64_t* tar_is_gt,
                       const int* chosen, const int* n_chosen, int max_num, const int64_t* labels,
                       long long label_ld, const float* boxes, long long box_ld, const b2d_pyramid* pyr_host,
                       const float* gt, int gt_ld, const int* gt_count, const int64_t* gt_label, int prepend_gt,
                       const float* means_host, const float* stds_host, int B, void* stream) {
    B2D_REQUIRE(chosen && n_chosen && labels && gt && gt_count, "encode_targets: null pointer");
    B2D_REQUIRE(boxes || pyr_host, "encode_targets: need boxes or pyramid");
    EncArgs p;
    p.chosen = chosen; p.n_chosen = n_chosen; p.max_num = max_num; p.labels = labels; p.label_ld = label_ld;
    p.boxes = boxes; p.box_ld = box_ld; p.use_pyr = boxes ? 0 : 1;
    p.gt = gt; p.gt_ld = gt_ld; p.gt_count = gt_count; p.gt_label = gt_label; p.prepend_gt = prepend_gt;
    for (int i = 0; i < 4; ++i) { p.ms[i] = means_host ? means_host[i] : 0.0f; p.ms[4 + i] = stds_host ? stds_host[i] : 1.0f; }
    b2d_pyramid pyr;
    memset(&pyr, 0, sizeof(pyr));
    if (p.use_pyr) pyr = *pyr_host;
    dim3 grid(cdiv(max_num, 128), B);
    k_encode_targets<<<grid, 128, 0, (cudaStream_t)stream>>>(p, pyr, tar_box, tar_gt, tar_param, tar_label, tar_is_gt);
    return check_launch("encode_targets");
}

int b2d_roi_targets_fused(int64_t* labels, float* max_iou, long long out_ld, const float* boxes, long long box_ld,
                          const int* box_count, long long N, const float* gt, int gt_ld, const int* gt_count,
                          const int64_t* gt_label, int B, float pos_iou, float neg_iou, float min_pos_iou,
                          int prepend_gt, int* census, int* pos_list, int pos_cap, int* chosen, int* n_chosen,
                          int max_num, int pos_num, unsigned long long seed, const unsigned long long* seed_step,
                          float* tar_box, float* tar_gt, float* tar_param, int64_t* tar_label, int64_t* tar_is_gt,
                          const float* means_host, const float* stds_host, void* stream) {
    B2D_REQUIRE(labels && max_iou && boxes && gt && gt_count && census && chosen && n_chosen, "roi_targets_fused: null pointer");
    B2D_REQUIRE(B >= 1 && gt_ld >= 1 && gt_ld <= kGtChunk && N >= 0 && N <= kSmallThreads * kSmallBoxes,
                "roi_targets_fused: need N <= 4096 and gt_ld <= 512");
    B2D_REQUIRE(max_num >= 1 && max_num <= kSmallThreads && pos_num >= 0 && pos_num <= max_num,
                "roi_targets_fused: need 1 <= max_num <= 1024 and pos_num <= max_num");
    AssignArgs a;
    a.boxes = boxes; a.box_ld = box_ld; a.box_count = box_count; a.N = N;
    a.use_pyr = 0; a.img_hw = nullptr; a.border = 0.0f;
    a.gt = gt; a.gt_ld = gt_ld; a.gt_count = gt_count;
    a.pos_iou = pos_iou; a.neg_iou = neg_iou; a.min_pos_iou = min_pos_iou;
    a.prepend_gt = prepend_gt; a.out_ld = out_ld;
    FusedArgs f;
    f.chosen = chosen; f.n_chosen = n_chosen; f.max_num = max_num; f.pos_num = pos_num; f.seed = seed; f.seed_step = seed_step;
    f.gt_label = gt_label;
    f.tar_box = tar_box; f.tar_gt = tar_gt; f.tar_param = tar_param; f.tar_label = tar_label; f.tar_is_gt = tar_is_gt;
    for (int i = 0; i < 4; ++i) { f.ms[i] = means_host ? means_host[i] : 0.0f; f.ms[4 + i] = stds_host ? stds_host[i] : 1.0f; }
    if (knobs().pdl) {
        // set up while the stream predecessor (the proposal kernel, which calls pdl_launch_dependents) still runs
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim = dim3((unsigned)B, 1, 1); cfg.blockDim = dim3(kSmallThreads, 1, 1); cfg.stream = (cudaStream_t)stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        const cudaError_t e = cudaLaunchKernelEx(&cfg, k_roi_targets_small, a, labels, max_iou, census, pos_list, pos_cap, f);
        if (e != cudaSuccess) { set_error(cudaGetErrorString(e)); cudaGetLastError(); return (int)e; }
    } else {
        k_roi_targets_small<<<B, kSmallThreads, 0, (cudaStream_t)stream>>>(a, labels, max_iou, census, pos_list, pos_cap, f);
    }
    return check_launch("roi_targets_fused");
}

}  // extern "C"
