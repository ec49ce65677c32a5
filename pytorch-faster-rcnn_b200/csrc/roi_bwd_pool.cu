// roi_bwd_pool.cu -- K6: atomic-free, deterministic RoIAlign backward; K7: RoIPool.
//
// K6 is formulated as a destination-ordered gather: the feature-gradient cells are
// the owners; each CTA owns a tile of cells of one (image, level) and walks the RoIs
// in ascending order, so every cell receives its contributions in exactly the order
// torchvision's sequential CPU kernel adds them (RoI, ph, pw, iy, ix, tap) --
// no atomics, no zero-fill pass (cells without contributions are written as 0), and
// bit-identical to the CPU reference.  RoIs are bucketed per tile by an ordered
// ballot compaction (the "sorted scatter" of the RoI list by destination tile).
//
// K7 follows torchvision.ops.roi_pool (rounded bounds, floor/ceil bins, argmax);
// its backward is a per-cell ordered gather over the argmax table.
#include <cstdlib>
#include <cstring>

#include "roi_bwd_common.cuh"

namespace b2d {

// roi_align_bwd_tile.cu
size_t roi_align_bwd_tile_workspace(long long R, int B, int L);
// patch form (roi_align_bwd_patch.cu): its workspace begins with the tile form's tables, so either can use it
size_t roi_align_bwd_patch_workspace(long long R, int B, const b2d_roi_cfg& c);
int roi_align_bwd_patch_try(void* const* grad_feat_ptrs_host, const RoiSets& q, const int* levels, long long R, int B,
                            const b2d_roi_cfg& c, void* workspace, cudaStream_t st);
int roi_align_bwd_tile_try(void* const* grad_feat_ptrs_host, const RoiSets& q, const int* levels, long long R, int B,
                           const b2d_roi_cfg& c, void* workspace, cudaStream_t st);

struct AxisTapB { int lo, hi; float l, h; int valid; };

__device__ __forceinline__ AxisTapB axis_tap_b(float start, float bin, int p, int i, int grid, int size) {
    AxisTapB t;
    float v = start + (float)p * bin + ((float)i + 0.5f) * bin / (float)grid;
    t.valid = !(v < -1.0f || v > (float)size);
    if (v <= 0.0f) v = 0.0f;
    int lo = (int)v, hi;
    if (lo >= size - 1) { hi = lo = size - 1; v = (float)lo; } else hi = lo + 1;
    t.lo = lo; t.hi = hi; t.l = v - (float)lo; t.h = 1.0f - t.l;
    return t;
}

constexpr int kTileH = 8, kTileW = 32;      // cells per CTA (one thread per cell)
constexpr int kChPerCta = 16;               // channels accumulated per thread
constexpr int kSub = 32;                    // RoIs per shared-memory batch
constexpr int kAxisMax = 16;                // PH*sr, PW*sr limit (7*2 = 14)

struct BwdArgs {
    b2d_roi_cfg cfg;
    void* grad[kMaxLevels];
    RoiSets q;
    const int* levels;                      // level of every slot, -1 = empty batched slot
    long long R; int B;
    int tile_off[kMaxLevels + 1];           // CTA-tile prefix per level (per image)
    int tiles_x[kMaxLevels];
};

// level of every slot of the batched entries, -1 for the slots at or past their image's count (their boxes unread)
__global__ void __launch_bounds__(256) k_bwd_levels_batched(int* __restrict__ lv, RoiSets q, long long R, float finest, int L) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    const RoiSlot sl = roi_slot(q, r);
    lv[r] = sl.box ? roi_level(sl.box[0], sl.box[sl.ld], sl.box[2 * sl.ld], sl.box[3 * sl.ld], finest, L) : -1;
}

__global__ void __launch_bounds__(256) k_roi_align_bwd(BwdArgs a) {
    __shared__ int s_list[kSub];
    __shared__ AxisTapB s_ty[kSub][kAxisMax], s_tx[kSub][kAxisMax];
    __shared__ int s_n, s_warp[8];
    __shared__ long long s_next;
    const b2d_roi_cfg& c = a.cfg;
    const int tiles_per_img = a.tile_off[c.num_levels];
    const int img = blockIdx.x / tiles_per_img;
    int t = blockIdx.x - img * tiles_per_img, lvl = 0;
    for (int q = 1; q < c.num_levels; ++q) if (t >= a.tile_off[q]) lvl = q;
    t -= a.tile_off[lvl];
    const int H = c.H[lvl], W = c.W[lvl];
    const int ty0 = (t / a.tiles_x[lvl]) * kTileH, tx0 = (t % a.tiles_x[lvl]) * kTileW;
    const int y = ty0 + (int)threadIdx.x / kTileW, x = tx0 + (int)threadIdx.x % kTileW;
    const bool live = y < H && x < W;
    const int c0 = blockIdx.y * kChPerCta;
    const int nch = min(kChPerCta, c.C - c0);
    const int bins = c.PH * c.PW, gy = c.sampling_ratio, gx = c.sampling_ratio;
    const int ny = c.PH * gy, nx = c.PW * gx;
    const float cnt = (float)max(gy * gx, 1);
    const float scale = c.spatial_scale[lvl];
    float acc[kChPerCta];
#pragma unroll
    for (int q = 0; q < kChPerCta; ++q) acc[q] = 0.0f;

    long long r0 = 0;
    while (true) {
        // ---- fill the batch with the next RoIs (ascending r) that can touch this tile
        if (threadIdx.x == 0) s_n = 0;
        __syncthreads();
        while (r0 < a.R && s_n < kSub) {
            const long long r = r0 + threadIdx.x;
            bool hit = false;
            const RoiSlot sl = r < a.R && a.levels[r] == lvl ? roi_slot(a.q, r) : RoiSlot{nullptr, 0, -1};
            if (sl.img == img) {
                const float off = c.aligned ? 0.5f : 0.0f;
                const float sx = sl.box[0] * scale - off, sy = sl.box[sl.ld] * scale - off;
                const float ex = sl.box[2 * sl.ld] * scale - off, ey = sl.box[3 * sl.ld] * scale - off;
                // conservative extent of the taps: samples lie in [s, max(e, s+1)], taps reach one cell
                // further, and everything beyond the map is clamped onto the last row / column
                float ylo = floorf(fminf(sy, ey)) - 1.0f, yhi = ceilf(fmaxf(ey, sy + 1.0f)) + 1.0f;
                float xlo = floorf(fminf(sx, ex)) - 1.0f, xhi = ceilf(fmaxf(ex, sx + 1.0f)) + 1.0f;
                ylo = fminf(ylo, (float)(H - 1)); xlo = fminf(xlo, (float)(W - 1));
                hit = !(yhi < (float)ty0 || ylo > (float)(ty0 + kTileH - 1) || xhi < (float)tx0 ||
                        xlo > (float)(tx0 + kTileW - 1));
            }
            const unsigned m = __ballot_sync(0xffffffffu, hit);
            if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = __popc(m);
            if (threadIdx.x == 0) s_next = r0 + blockDim.x;
            __syncthreads();
            int before = s_n;
            for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) before += s_warp[w];
            const int pos = before + __popc(m & ((1u << (threadIdx.x & 31)) - 1u));
            if (hit) {
                if (pos < kSub) s_list[pos] = (int)r;
                else if (pos == kSub) s_next = r;          // first RoI that did not fit: resume there
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                int tot = s_n;
                for (int w = 0; w < 8; ++w) tot += s_warp[w];
                s_n = min(tot, kSub);
            }
            __syncthreads();
            r0 = s_next;
        }
        const int nb = s_n;
        if (nb == 0) break;
        // ---- axis taps of the batch
        for (int q = threadIdx.x; q < nb * (ny + nx); q += blockDim.x) {
            const int e = q / (ny + nx), k = q - e * (ny + nx);
            const RoiSlot sl = roi_slot(a.q, s_list[e]);
            const float* rp = sl.box;
            const float off = c.aligned ? 0.5f : 0.0f;
            const float sx = rp[0] * scale - off, sy = rp[sl.ld] * scale - off;
            const float ex = rp[2 * sl.ld] * scale - off, ey = rp[3 * sl.ld] * scale - off;
            float rw = ex - sx, rh = ey - sy;
            if (!c.aligned) { rw = fmaxf(rw, 1.0f); rh = fmaxf(rh, 1.0f); }
            const float bh = rh / (float)c.PH, bw = rw / (float)c.PW;
            if (k < ny) s_ty[e][k] = axis_tap_b(sy, bh, k / gy, k % gy, gy, H);
            else s_tx[e][k - ny] = axis_tap_b(sx, bw, (k - ny) / gx, (k - ny) % gx, gx, W);
        }
        __syncthreads();
        // ---- ordered accumulation
        if (live) {
            for (int e = 0; e < nb; ++e) {
                const float* go = gout_row(a.q, s_list[e], (long long)c.C * bins) + (long long)c0 * bins;
                for (int ph = 0; ph < c.PH; ++ph) {
                    // does any y-sample of this bin row touch row y?
                    bool anyy = false;
                    for (int iy = 0; iy < gy; ++iy) { const AxisTapB ty = s_ty[e][ph * gy + iy]; anyy |= ty.valid && (ty.lo == y || ty.hi == y); }
                    if (!anyy) continue;
                    for (int pw = 0; pw < c.PW; ++pw) {
                        bool anyx = false;
                        for (int ix = 0; ix < gx; ++ix) { const AxisTapB tx = s_tx[e][pw * gx + ix]; anyx |= tx.valid && (tx.lo == x || tx.hi == x); }
                        if (!anyx) continue;
                        const int bin = ph * c.PW + pw;
                        for (int iy = 0; iy < gy; ++iy) {
                            const AxisTapB ty = s_ty[e][ph * gy + iy];
                            for (int ix = 0; ix < gx; ++ix) {
                                const AxisTapB tx = s_tx[e][pw * gx + ix];
                                if (!(ty.valid && tx.valid)) continue;
                                const float w[4] = {ty.h * tx.h, ty.h * tx.l, ty.l * tx.h, ty.l * tx.l};
                                const bool m[4] = {ty.lo == y && tx.lo == x, ty.lo == y && tx.hi == x,
                                                   ty.hi == y && tx.lo == x, ty.hi == y && tx.hi == x};
#pragma unroll
                                for (int k = 0; k < 4; ++k) {
                                    if (!m[k]) continue;
#pragma unroll
                                    for (int q = 0; q < kChPerCta; ++q)
                                        if (q < nch) acc[q] += __ldg(go + (long long)q * bins + bin) * w[k] / cnt;
                                }
                            }
                        }
                    }
                }
            }
        }
        __syncthreads();
    }
    if (live) {
        float* g = reinterpret_cast<float*>(a.grad[lvl]);
        if (c.layout == 0) {
#pragma unroll
            for (int q = 0; q < kChPerCta; ++q)
                if (q < nch) g[(((long long)img * c.C + c0 + q) * H + y) * W + x] = acc[q];
        } else {
#pragma unroll
            for (int q = 0; q < kChPerCta; ++q)
                if (q < nch) g[(((long long)img * H + y) * W + x) * c.C + c0 + q] = acc[q];
        }
    }
}

// ------------------------------------------------------------------ K7 RoIPool
__global__ void __launch_bounds__(256) k_roi_pool_fwd(float* __restrict__ out, int* __restrict__ argmax,
                                                      const float* __restrict__ feat, int C, int H, int W,
                                                      const float* __restrict__ rois, long long ld,
                                                      const int* __restrict__ roi_img, long long R, float scale,
                                                      int PH, int PW) {
    const long long total = R * C * PH * PW;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const int pw = (int)(t % PW), ph = (int)((t / PW) % PH);
    const int ch = (int)((t / ((long long)PW * PH)) % C);
    const long long r = t / ((long long)PW * PH * C);
    const int img = roi_img ? roi_img[r] : 0;
    const int sw = (int)roundf(rois[r] * scale), sh = (int)roundf(rois[ld + r] * scale);
    const int ew = (int)roundf(rois[2 * ld + r] * scale), eh = (int)roundf(rois[3 * ld + r] * scale);
    const int rw = max(ew - sw + 1, 1), rh = max(eh - sh + 1, 1);
    const float bh = (float)rh / (float)PH, bw = (float)rw / (float)PW;
    int hs = (int)floorf((float)ph * bh), ws = (int)floorf((float)pw * bw);
    int he = (int)ceilf((float)(ph + 1) * bh), we = (int)ceilf((float)(pw + 1) * bw);
    hs = min(max(hs + sh, 0), H); he = min(max(he + sh, 0), H);
    ws = min(max(ws + sw, 0), W); we = min(max(we + sw, 0), W);
    const bool empty = (he <= hs) || (we <= ws);
    const float* f = feat + ((long long)img * C + ch) * H * W;
    float mv = empty ? 0.0f : -3.402823466e+38F;
    int mi = -1;
    for (int h = hs; h < he; ++h)
        for (int w = ws; w < we; ++w) {
            const float v = __ldg(f + h * W + w);
            if (v > mv) { mv = v; mi = h * W + w; }
        }
    out[t] = mv;
    argmax[t] = mi;
}

// one thread per feature cell (img, c, h, w); RoIs visited in ascending order
__global__ void __launch_bounds__(256) k_roi_pool_bwd(float* __restrict__ grad, const float* __restrict__ gout,
                                                      const int* __restrict__ argmax, int B, int C, int H, int W,
                                                      const float* __restrict__ rois, long long ld,
                                                      const int* __restrict__ roi_img, long long R, float scale,
                                                      int PH, int PW) {
    extern __shared__ __align__(16) int s_roi[];             // per RoI: sh, sw, rh, rw, img  (chunks of 256)
    const long long total = (long long)B * C * H * W;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = t < total;
    const int w = (int)(t % W), h = (int)((t / W) % H);
    const int ch = (int)((t / ((long long)W * H)) % C), img = (int)(t / ((long long)W * H * C));
    float acc = 0.0f;
    for (long long r0 = 0; r0 < R; r0 += 256) {
        __syncthreads();
        const long long r = r0 + threadIdx.x;
        if (r < R) {
            const int sw = (int)roundf(rois[r] * scale), sh = (int)roundf(rois[ld + r] * scale);
            const int ew = (int)roundf(rois[2 * ld + r] * scale), eh = (int)roundf(rois[3 * ld + r] * scale);
            s_roi[threadIdx.x * 5 + 0] = sh; s_roi[threadIdx.x * 5 + 1] = sw;
            s_roi[threadIdx.x * 5 + 2] = max(eh - sh + 1, 1); s_roi[threadIdx.x * 5 + 3] = max(ew - sw + 1, 1);
            s_roi[threadIdx.x * 5 + 4] = roi_img ? roi_img[r] : 0;
        }
        __syncthreads();
        if (!live) continue;
        const int nb = (int)min((long long)256, R - r0);
        for (int e = 0; e < nb; ++e) {
            if (s_roi[e * 5 + 4] != img) continue;
            const int sh = s_roi[e * 5], sw = s_roi[e * 5 + 1], rh = s_roi[e * 5 + 2], rw = s_roi[e * 5 + 3];
            if (h < sh - 1 || h > sh + rh || w < sw - 1 || w > sw + rw) continue;
            const float bh = (float)rh / (float)PH, bw = (float)rw / (float)PW;
            const long long ob = ((r0 + e) * C + ch) * PH * PW;
            for (int ph = 0; ph < PH; ++ph) {
                int hs = (int)floorf((float)ph * bh) + sh, he = (int)ceilf((float)(ph + 1) * bh) + sh;
                hs = min(max(hs, 0), H); he = min(max(he, 0), H);
                if (h < hs || h >= he) continue;
                for (int pw = 0; pw < PW; ++pw) {
                    int ws = (int)floorf((float)pw * bw) + sw, we = (int)ceilf((float)(pw + 1) * bw) + sw;
                    ws = min(max(ws, 0), W); we = min(max(we, 0), W);
                    if (w < ws || w >= we) continue;
                    if (argmax[ob + ph * PW + pw] == h * W + w) acc += gout[ob + ph * PW + pw];
                }
            }
        }
    }
    if (live) grad[t] = acc;
}

}  // namespace b2d

using namespace b2d;

extern "C" {

static size_t bwd_levels_bytes(long long R) { return (((size_t)(R > 0 ? R : 1) * 4 + 256) + 255) & ~(size_t)255; }

size_t b2d_roi_align_bwd_workspace_bytes(long long R, int B, const b2d_roi_cfg* cfg_host) {
    const int L = cfg_host ? cfg_host->num_levels : B2D_MAX_LEVELS;
    size_t n = roi_align_bwd_tile_workspace(R, B > 0 ? B : 1, L);                     // tile-kernel tables
    if (cfg_host && cfg_host->layout == 1 && cfg_host->sampling_ratio == 2 && cfg_host->num_levels >= 1 &&
        cfg_host->num_levels <= B2D_MAX_LEVELS) {
        const size_t p = roi_align_bwd_patch_workspace(R, B > 0 ? B : 1, *cfg_host);  // + bitmaps + patch scratch
        if (p > n) n = p;
    }
    return bwd_levels_bytes(R) + n;                                                   // level ids in front
}

// the entry points below: an explicit RoI list with roi_img / levels, or the image-major [B][4][ld] slots of
// b2d_roi_align_fwd_batched with per-image counts, one or several sets of them (RoiSets)
static int roi_align_bwd_impl(void* const* grad_feat_ptrs_host, const RoiSets& q, const int* levels, long long R, int B,
                              const b2d_roi_cfg* cfg_host, void* workspace, size_t ws_bytes, void* stream) {
    B2D_REQUIRE(grad_feat_ptrs_host && cfg_host && R >= 0 && B >= 1, "roi_align_bwd: bad args");
    const b2d_roi_cfg& c = *cfg_host;
    B2D_REQUIRE(c.num_levels >= 1 && c.num_levels <= B2D_MAX_LEVELS, "roi_align_bwd: bad cfg");
    B2D_REQUIRE(c.layout == 0 || c.layout == 1, "roi_align_bwd: fp32 NCHW (0) or NHWC (1) gradients only");
    B2D_REQUIRE(c.sampling_ratio > 0 && c.PH * c.sampling_ratio <= kAxisMax && c.PW * c.sampling_ratio <= kAxisMax,
                "roi_align_bwd: needs a fixed sampling_ratio with PH*sr, PW*sr <= 16");
    B2D_REQUIRE(workspace && ws_bytes >= b2d_roi_align_bwd_workspace_bytes(R, B, cfg_host), "roi_align_bwd: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    {   // NHWC fp32 gradients with 2x2 samples: patch form (B2D_ROI_BWD_TILE=2, default), tile-gather form (=1);
        // B2D_ROI_BWD_TILE=0 forces the generic, torchvision-bit-identical kernel below
        if (knobs().roi_bwd_tile >= 2) {                  // patch form ("sorted scatter", roi_align_bwd_patch.cu): default
            const int rc = roi_align_bwd_patch_try(grad_feat_ptrs_host, q, levels, R, B, c, (char*)workspace + bwd_levels_bytes(R), st);
            if (rc != 1) return rc;
        }
        if (knobs().roi_bwd_tile != 0) {
            const int rc = roi_align_bwd_tile_try(grad_feat_ptrs_host, q, levels, R, B, c, (char*)workspace + bwd_levels_bytes(R), st);
            if (rc != 1) return rc;
        }
    }
    int* lv = (int*)workspace;
    if (q.ld[0] > 0) {
        if (R > 0) k_bwd_levels_batched<<<cdiv(R, 256), 256, 0, st>>>(lv, q, R, c.finest_scale, c.num_levels);
    } else if (levels) {
        cudaMemcpyAsync(lv, levels, sizeof(int) * R, cudaMemcpyDeviceToDevice, st);
    } else if (R > 0) {
        int rc = b2d_roi_levels(lv, q.rois[0], q.roi_ld, R, c.finest_scale, c.num_levels, stream);
        if (rc != B2D_OK) return rc;
    }
    BwdArgs a;
    memset(&a, 0, sizeof(a));
    a.cfg = c;
    int run = 0;
    for (int l = 0; l < c.num_levels; ++l) {
        a.grad[l] = grad_feat_ptrs_host[l];
        a.tile_off[l] = run;
        a.tiles_x[l] = cdiv(c.W[l], kTileW);
        run += a.tiles_x[l] * cdiv(c.H[l], kTileH);
    }
    a.tile_off[c.num_levels] = run;
    a.q = q; a.levels = lv; a.R = R; a.B = B;
    dim3 grid((unsigned)(run * B), cdiv(c.C, kChPerCta));
    k_roi_align_bwd<<<grid, 256, 0, st>>>(a);
    return check_launch("roi_align_bwd");
}

int b2d_roi_align_bwd(void* const* grad_feat_ptrs_host, const float* grad_out, const float* rois, long long roi_ld,
                      const int* roi_img, const int* levels, long long R, int B, const b2d_roi_cfg* cfg_host,
                      void* workspace, size_t ws_bytes, void* stream) {
    B2D_REQUIRE(grad_out && rois, "roi_align_bwd: bad args");
    RoiSets q;
    memset(&q, 0, sizeof(q));
    q.S = 1; q.roi_ld = roi_ld; q.roi_img = roi_img; q.base[1] = R; q.rois[0] = rois; q.gout[0] = grad_out;
    return roi_align_bwd_impl(grad_feat_ptrs_host, q, levels, R, B, cfg_host, workspace, ws_bytes, stream);
}

// slots of S batched sets (0 if the arguments are out of range: the entry then refuses them)
static long long multi_slots(int S, const long long* ld_host, int B) {
    if (S < 1 || S > kMaxSets || !ld_host || B < 1) return 0;
    long long R = 0;
    for (int s = 0; s < S; ++s) {
        if (ld_host[s] < 1) return 0;
        R += ld_host[s] * B;
    }
    return R;
}

size_t b2d_roi_align_bwd_multi_workspace_bytes(int S, const long long* ld_host, int B, const b2d_roi_cfg* cfg_host) {
    return b2d_roi_align_bwd_workspace_bytes(multi_slots(S, ld_host, B), B, cfg_host);
}

int b2d_roi_align_bwd_multi(void* const* grad_feat_ptrs_host, int S, const float* const* grad_out_host,
                            const float* const* rois_host, const long long* ld_host, const int* const* counts_host, int B,
                            const b2d_roi_cfg* cfg_host, void* workspace, size_t ws_bytes, void* stream) {
    const long long R = multi_slots(S, ld_host, B);
    B2D_REQUIRE(R > 0 && grad_out_host && rois_host && counts_host, "roi_align_bwd_multi: bad args (1 <= S <= 4, ld >= 1, B >= 1)");
    RoiSets q;
    memset(&q, 0, sizeof(q));
    q.S = S;
    for (int s = 0; s < S; ++s) {
        B2D_REQUIRE(grad_out_host[s] && rois_host[s] && counts_host[s], "roi_align_bwd_multi: NULL set pointer");
        q.ld[s] = ld_host[s]; q.rois[s] = rois_host[s]; q.gout[s] = grad_out_host[s]; q.counts[s] = counts_host[s];
        q.base[s + 1] = q.base[s] + ld_host[s] * B;
    }
    return roi_align_bwd_impl(grad_feat_ptrs_host, q, nullptr, R, B, cfg_host, workspace, ws_bytes, stream);
}

size_t b2d_roi_align_bwd_batched_workspace_bytes(long long ld, int B, const b2d_roi_cfg* cfg_host) {
    return b2d_roi_align_bwd_multi_workspace_bytes(1, &ld, B, cfg_host);
}

int b2d_roi_align_bwd_batched(void* const* grad_feat_ptrs_host, const float* grad_out, const float* rois, long long ld,
                              const int* counts, int B, const b2d_roi_cfg* cfg_host, void* workspace, size_t ws_bytes,
                              void* stream) {
    return b2d_roi_align_bwd_multi(grad_feat_ptrs_host, 1, &grad_out, &rois, &ld, &counts, B, cfg_host, workspace, ws_bytes,
                                   stream);
}

int b2d_roi_pool_fwd(float* out, int* argmax, const float* feat, int B, int C, int H, int W, const float* rois,
                     long long roi_ld, const int* roi_img, long long R, float spatial_scale, int PH, int PW,
                     void* stream) {
    B2D_REQUIRE(out && argmax && feat && rois && B >= 1 && C >= 1 && R >= 0, "roi_pool_fwd: bad args");
    const long long total = R * C * PH * PW;
    if (total == 0) return B2D_OK;
    k_roi_pool_fwd<<<cdiv(total, 256), 256, 0, (cudaStream_t)stream>>>(out, argmax, feat, C, H, W, rois, roi_ld, roi_img, R,
                                                                      spatial_scale, PH, PW);
    return check_launch("roi_pool_fwd");
}

int b2d_roi_pool_bwd(float* grad_feat, const float* grad_out, const int* argmax, int B, int C, int H, int W,
                     const float* rois, long long roi_ld, const int* roi_img, long long R, float spatial_scale,
                     int PH, int PW, void* workspace, size_t ws_bytes, void* stream) {
    (void)workspace; (void)ws_bytes;
    B2D_REQUIRE(grad_feat && grad_out && argmax && rois && B >= 1 && C >= 1 && R >= 0, "roi_pool_bwd: bad args");
    const long long total = (long long)B * C * H * W;
    if (total == 0) return B2D_OK;
    k_roi_pool_bwd<<<cdiv(total, 256), 256, 256 * 5 * sizeof(int), (cudaStream_t)stream>>>(
        grad_feat, grad_out, argmax, B, C, H, W, rois, roi_ld, roi_img, R, spatial_scale, PH, PW);
    return check_launch("roi_pool_bwd");
}

}  // extern "C"
