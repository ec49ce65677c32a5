// roi_common.cuh -- RoI argument block, RoI fetch, FPN level map and the bilinear sample geometry
// shared by the RoIAlign forward (roi_align.cu), its backward (roi_bwd_common.cuh) and the sparse
// feature fetch (roi_fetch.cu).  torchvision RoIAlign semantics (pre_calc_for_bilinear_interpolate);
// lib/region.py:243-306.
#pragma once
#include "common.cuh"

namespace b2d {

struct RoiArgs {
    b2d_roi_cfg cfg;
    const void* feat[kMaxLevels];
    const float* rois; long long roi_ld;
    const int* roi_img; const int* levels;
    long long R;
    long long batched_ld;          // > 0: rois are image-major [B][4][ld], counts per image
    const int* counts;
};

// slot r -> (image, coordinates); false if the slot is past the image's count
__device__ __forceinline__ bool roi_fetch(const RoiArgs& a, long long r, int& img, float& x1, float& y1, float& x2,
                                          float& y2) {
    if (a.batched_ld > 0) {
        img = (int)(r / a.batched_ld);
        const long long i = r - (long long)img * a.batched_ld;
        if (i >= a.counts[img]) return false;
        const float* p = a.rois + (long long)img * 4 * a.batched_ld + i;
        x1 = p[0]; y1 = p[a.batched_ld]; x2 = p[2 * a.batched_ld]; y2 = p[3 * a.batched_ld];
        return true;
    }
    img = a.roi_img ? a.roi_img[r] : 0;
    x1 = a.rois[r]; y1 = a.rois[a.roi_ld + r]; x2 = a.rois[2 * a.roi_ld + r]; y2 = a.rois[3 * a.roi_ld + r];
    return true;
}

__device__ __forceinline__ int roi_level(const float x1, const float y1, const float x2, const float y2,
                                         float finest, int num_levels) {
    // lib/region.py:256-264
    const float s = sqrtf(((x2 - x1) + 1.0f) * ((y2 - y1) + 1.0f));
    float t = floorf(log2f(s / finest + 1e-6f));
    t = fminf(fmaxf(t, 0.0f), (float)(num_levels - 1));
    return (int)t;
}

// One axis of the sample grid of one RoI (torchvision pre_calc_for_bilinear_interpolate).
struct AxisTap { int lo, hi; float l, h; int valid; };

__device__ __forceinline__ AxisTap axis_tap(float start, float bin, int p, int i, int grid, int size) {
    AxisTap t;
    float v = start + (float)p * bin + ((float)i + 0.5f) * bin / (float)grid;
    t.valid = !(v < -1.0f || v > (float)size);
    if (v <= 0.0f) v = 0.0f;
    int lo = (int)v, hi;
    if (lo >= size - 1) { hi = lo = size - 1; v = (float)lo; } else hi = lo + 1;
    t.lo = lo; t.hi = hi;
    t.l = v - (float)lo; t.h = 1.0f - t.l;
    return t;
}

struct RoiGeom { float sx, sy, bw, bh; int gx, gy; };

__device__ __forceinline__ RoiGeom roi_geom(float x1, float y1, float x2, float y2, float scale, int PH, int PW,
                                            int sr, int aligned) {
    RoiGeom g;
    const float off = aligned ? 0.5f : 0.0f;
    g.sx = x1 * scale - off; g.sy = y1 * scale - off;
    const float ex = x2 * scale - off, ey = y2 * scale - off;
    float rw = ex - g.sx, rh = ey - g.sy;
    if (!aligned) { rw = fmaxf(rw, 1.0f); rh = fmaxf(rh, 1.0f); }
    g.bh = rh / (float)PH; g.bw = rw / (float)PW;
    g.gy = sr > 0 ? sr : (int)ceilf(rh / (float)PH);
    g.gx = sr > 0 ? sr : (int)ceilf(rw / (float)PW);
    return g;
}

}  // namespace b2d
