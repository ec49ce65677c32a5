// roi_bwd_common.cuh -- per-RoI geometry record and the (image, level) bucket lists shared by the two NHWC RoIAlign
// backward forms (roi_align_bwd_tile.cu: tile gather; roi_align_bwd_patch.cu: per-RoI patches + ordered merge).
#pragma once
#include "roi_common.cuh"

namespace b2d {

constexpr int kMaxS = 16;              // samples per axis (PH * 2, PW * 2 <= 16)
constexpr int kMaxBinsT = 64;

struct __align__(16) BwdMeta {
    int img, lvl, y0, y1;
    int x0, x1; float sx, sy;
    float bw, bh; int _p0, _p1;
};

constexpr int kMaxSets = 4;            // RoI sets of one b2d_roi_align_bwd_multi call

// The RoI slots of one K6 call.  Batched entries: S sets, set s the image-major [B][4][ld[s]] list b2d_roi_align_fwd_batched
// read for it, with counts[s][B]; slots are numbered set-major, r = base[s] + b * ld[s] + j, and the grad_out row of slot r
// is row b * ld[s] + j of gout[s].  Bucket lists are ascending in r, so a cell adds its contributions set by set: the result
// is that of the unbatched entry on the compacted lists concatenated set-major.  The unbatched entry is one set with
// ld[0] = 0: slot r is column r of rois[0] (stride roi_ld), of image roi_img[r], with grad_out row r.
struct RoiSets {
    int S;
    long long roi_ld;
    const int* roi_img;
    long long base[kMaxSets + 1];      // first slot of each set; base[S] = R
    long long ld[kMaxSets];
    const float* rois[kMaxSets];
    const float* gout[kMaxSets];
    const int* counts[kMaxSets];
};

__device__ __forceinline__ int set_of(const RoiSets& q, long long r) {
    int s = 0;
    while (s + 1 < q.S && r >= q.base[s + 1]) ++s;
    return s;
}

// first float of the grad_out row of slot r (`row` = C * PH * PW floats per row)
__device__ __forceinline__ const float* gout_row(const RoiSets& q, long long r, long long row) {
    const int s = set_of(q, r);
    return q.gout[s] + (r - q.base[s]) * row;
}

struct RoiSlot { const float* box; long long ld; int img; };      // box: x1, coordinate k at box[k * ld]

// box and image of slot r; box = NULL for a batched slot at or past its image's count (its box is not read)
__device__ __forceinline__ RoiSlot roi_slot(const RoiSets& q, long long r) {
    RoiSlot o;
    const int s = set_of(q, r);
    const long long ld = q.ld[s];
    if (ld == 0) {
        o.box = q.rois[0] + r; o.ld = q.roi_ld; o.img = q.roi_img ? q.roi_img[r] : 0;
        return o;
    }
    const long long k = r - q.base[s];
    o.img = (int)(k / ld);
    const long long j = k - (long long)o.img * ld;
    o.box = j < q.counts[s][o.img] ? q.rois[s] + (long long)o.img * 4 * ld + j : nullptr;
    o.ld = ld;
    return o;
}

struct MetaArgs {
    b2d_roi_cfg cfg;
    RoiSets q;
    const int* levels;                 // unbatched entry only (NULL: the level map)
    long long R;
};

// The record of slot r.  A batched slot at or past its image's count gets img = -1 and an empty tap box: no bucket lists
// it and it has no patch, so neither its box nor its grad_out row is ever read.
__device__ __forceinline__ BwdMeta bwd_meta_of(const MetaArgs& a, long long r) {
    const b2d_roi_cfg& c = a.cfg;
    BwdMeta m;
    const RoiSlot sl = roi_slot(a.q, r);
    if (!sl.box) {
        m.img = -1; m.lvl = 0; m.y0 = m.x0 = 0; m.y1 = m.x1 = -1;
        m.sx = m.sy = m.bw = m.bh = 0.0f; m._p0 = m._p1 = 0;
        return m;
    }
    m.img = sl.img;
    const float* p = sl.box;
    const long long ld = sl.ld;
    const float x1 = p[0], y1 = p[ld], x2 = p[2 * ld], y2 = p[3 * ld];
    m.lvl = a.levels ? a.levels[r] : (c.num_levels > 1 ? roi_level(x1, y1, x2, y2, c.finest_scale, c.num_levels) : 0);
    const int H = c.H[m.lvl], W = c.W[m.lvl];
    const RoiGeom g = roi_geom(x1, y1, x2, y2, c.spatial_scale[m.lvl], c.PH, c.PW, 2, c.aligned);
    m.sx = g.sx; m.sy = g.sy; m.bw = g.bw; m.bh = g.bh;
    // cell bounding box of all taps (sample positions need not be monotone for malformed RoIs: take min / max)
    int y0 = H, y1c = -1, x0 = W, x1c = -1;
    for (int s = 0; s < 2 * c.PH; ++s) {
        const AxisTap t = axis_tap(g.sy, g.bh, s >> 1, s & 1, 2, H);
        if (t.valid) { y0 = min(y0, t.lo); y1c = max(y1c, t.hi); }
    }
    for (int s = 0; s < 2 * c.PW; ++s) {
        const AxisTap t = axis_tap(g.sx, g.bw, s >> 1, s & 1, 2, W);
        if (t.valid) { x0 = min(x0, t.lo); x1c = max(x1c, t.hi); }
    }
    m.y0 = y0; m.y1 = y1c; m.x0 = x0; m.x1 = x1c; m._p0 = m._p1 = 0;
    return m;
}

static __global__ void __launch_bounds__(256) k_bwd_meta(MetaArgs a, BwdMeta* __restrict__ meta) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= a.R) return;
    meta[r] = bwd_meta_of(a, r);
}

// bucket[(img * L + lvl) * R + k] = k-th RoI (ascending) of that feature map; bcount[img * L + lvl]
static __global__ void __launch_bounds__(256) k_bwd_bucket(const BwdMeta* __restrict__ meta, long long R, int L,
                                                    int* __restrict__ bucket, int* __restrict__ bcount) {
    __shared__ int s_warp[8], s_base;
    const int img = blockIdx.x / L, lvl = blockIdx.x - img * L;
    int* out = bucket + (long long)blockIdx.x * R;
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    for (long long r0 = 0; r0 < R; r0 += 256) {
        const long long r = r0 + threadIdx.x;
        const bool hit = r < R && meta[r].img == img && meta[r].lvl == lvl;
        const unsigned m = __ballot_sync(0xffffffffu, hit);
        if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = __popc(m);
        __syncthreads();
        int before = s_base;
        for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) before += s_warp[w];
        if (hit) out[before + __popc(m & ((1u << (threadIdx.x & 31)) - 1u))] = (int)r;
        __syncthreads();
        if (threadIdx.x == 0) { int t = 0; for (int w = 0; w < 8; ++w) t += s_warp[w]; s_base += t; }
        __syncthreads();
    }
    if (threadIdx.x == 0) bcount[blockIdx.x] = s_base;
}

}  // namespace b2d
