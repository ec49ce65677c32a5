// roi_align_bwd_tile.cu -- K6, tile-gather form: deterministic, atomic-free RoIAlign backward for NHWC fp32
// gradients and 2x2 samples per bin (every reference config).
//
// The first K6 (roi_bwd_pool.cu, k_roi_align_bwd: one thread per cell, every CTA scanning all RoIs and testing
// all 14 x 14 samples of each) is bit-identical to torchvision's CPU kernel but takes 41 ms at config-2/3 sizes
// (4096 RoIs x 256 channels: 23 GB/s).  Here the work is exactly the 784 taps of a RoI:
//   k_bwd_meta      per RoI: level, sample geometry, cell bounding box of its taps
//   k_bwd_bucket    per (image, level): the RoIs of that feature map, in ascending order ("sorted scatter" of the
//                   RoI list by destination, ordered ballot compaction)
//   k_roi_align_bwd_tile  one 512-thread CTA per (16 x 16 cell tile, 128-channel group).  For every RoI of the bucket that
//                   touches the tile (ascending): stage grad_out[roi][128 ch][bins] / 4 in shared memory as
//                   [bin][channel]; per tile row / column list the sample rows / columns whose taps hit it with
//                   their weights (hy or ly / hx or lx); then a thread (warp = tile row, lane = 4 channels) walks its 16 cells and adds
//                   sum_{(sy, wy) in row} sum_{(sx, wx) in col} (wy * wx) * g[bin(sy, sx)] -- the same per-tap terms
//                   as torchvision (grad / count * w), accumulated in registers in a fixed order.  Cells are owned
//                   by exactly one thread: no atomics, no zero-fill pass, run-to-run bit-identical.
// The summation order inside a cell differs from torchvision's sequential CPU order (RoI, ph, pw, iy, ix, tap), so
// the result is equal within rounding (1e-5 relative, the north_star tolerance), not bit-identical; the generic kernel
// remains for NCHW gradients / other sampling ratios.
// HBM roofline: grad_out read (50 176 B/RoI, ~4x from L2: a RoI overlaps ~4 tiles) + every gradient cell written once.
#include <cstring>

#include "roi_bwd_common.cuh"

namespace b2d {
namespace {

constexpr int kT = 16;                 // tile side in cells
constexpr int kCg = 128;               // channels per CTA
constexpr int kBT = 512;               // threads per CTA: warp w owns tile row w, lane l channels 4l .. 4l + 3
constexpr int kPitch = kCg + 4;        // shared-memory pitch of a bin row (floats)

struct TileArgs {
    b2d_roi_cfg cfg;
    float* grad[kMaxLevels];
    RoiSets q;                         // grad_out rows
    const BwdMeta* meta; const int* bucket; const int* bcount;
    long long R;
    int tile_off[kMaxLevels + 1], tiles_x[kMaxLevels];
    unsigned n_tiles;                  // tiles x images (grid.x of the ordinary launch)
    const int* guard;                  // non-NULL: run only if *guard != 0 (fallback of the patch form, roi_align_bwd_patch.cu)
};

struct __align__(8) ColTerm { float w; int off; };     // column weight, float offset of its bin column in s_g
constexpr size_t kTablesBytes = sizeof(float) * kT * kMaxS * 2 + sizeof(int) * kT * kMaxS * 2 + sizeof(ColTerm) * kT * kMaxS * 2 +
                                2 * sizeof(int) * kT;

__global__ void __launch_bounds__(kBT, 1) k_roi_align_bwd_tile(TileArgs a) {
    // Everything a RoI needs (staged gradients + tap tables) is double-buffered, so ONE barrier per RoI is enough:
    // a warp that is through with RoI e stages / tabulates RoI e + 1 into the other buffers while slower warps
    // still accumulate RoI e; the barrier of e + 1 is what protects the buffers of e from RoI e + 2.
    extern __shared__ __align__(16) char s_dyn[];
    struct Tables {
        float roww[kT][kMaxS * 2];
        int rowb[kT][kMaxS * 2];                         // float offset of the bin row in the staged block
        ColTerm col[kT][kMaxS * 2];
        int rown[kT], coln[kT];
    };
    float (*s_g)[kMaxBinsT * kPitch] = reinterpret_cast<float (*)[kMaxBinsT * kPitch]>(s_dyn);
    Tables* s_tab = reinterpret_cast<Tables*>(s_dyn + 2 * sizeof(float) * kMaxBinsT * kPitch);
    __shared__ int s_list[kBT], s_n, s_warp[kBT / 32];
    if (a.guard && *a.guard == 0) return;
    // one tile per CTA in the ordinary launch; the guarded fallback launch is persistent (a few CTAs per SM striding over
    // the tiles), so that it costs a microsecond when the guard says there is nothing to do
    for (unsigned bx = blockIdx.x; bx < a.n_tiles; bx += gridDim.x) {
    const b2d_roi_cfg& c = a.cfg;
    const int tiles_per_img = a.tile_off[c.num_levels];
    const int img = bx / tiles_per_img;
    int t = bx - img * tiles_per_img, lvl = 0;
    for (int q = 1; q < c.num_levels; ++q) if (t >= a.tile_off[q]) lvl = q;
    t -= a.tile_off[lvl];
    const int H = c.H[lvl], W = c.W[lvl], C = c.C, bins = c.PH * c.PW;
    const int ty0 = (t / a.tiles_x[lvl]) * kT, tx0 = (t % a.tiles_x[lvl]) * kT;
    const int cg = blockIdx.y;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int cq = lane;
    const int row = warp;                                // tile row owned by this warp (lane: 4 channels)
    float acc[kT][4];
#pragma unroll
    for (int x = 0; x < kT; ++x) { acc[x][0] = acc[x][1] = acc[x][2] = acc[x][3] = 0.0f; }
    // staging map of this thread: channel tid % 64, bins tid / 64 + 4 k (no index arithmetic in the loops; the 32 B
    // sectors a warp touches are re-used by its next 7 loads out of L1)
    constexpr int kStage = (kMaxBinsT + 3) / 4;
    const int sch = tid & (kCg - 1), sb0 = tid >> 7;
    float sv[kStage];

    const int* bl = a.bucket + (long long)(img * c.num_levels + lvl) * a.R;
    const int nb = a.bcount[img * c.num_levels + lvl];
    auto fetch = [&](int r) {                            // grad_out[r][cg * 64 .. + 64][bins] -> registers
        const float* go = gout_row(a.q, r, (long long)C * bins) + ((long long)cg * kCg + sch) * bins + sb0;
#pragma unroll
        for (int k = 0; k < kStage; ++k) sv[k] = (sb0 + 4 * k < bins) ? go[4 * k] : 0.0f;
    };
    auto stash = [&](float* dst) {                       // registers -> [bin][channel] / 4
        float* d = dst + sb0 * kPitch + sch;
#pragma unroll
        for (int k = 0; k < kStage; ++k)
            if (sb0 + 4 * k < bins) d[4 * k * kPitch] = sv[k] * 0.25f;
    };
    for (int base = 0; base < nb; base += kBT) {
        // ---- RoIs of this chunk whose taps touch the tile, ascending
        {
            const int k = base + tid;
            bool hit = false;
            int r = 0;
            if (k < nb) {
                r = bl[k];
                const BwdMeta m = a.meta[r];
                hit = !(m.y1 < ty0 || m.y0 > ty0 + kT - 1 || m.x1 < tx0 || m.x0 > tx0 + kT - 1);
            }
            const unsigned bm = __ballot_sync(0xffffffffu, hit);
            if (lane == 0) s_warp[warp] = __popc(bm);
            __syncthreads();
            int before = 0;
            for (int w = 0; w < warp; ++w) before += s_warp[w];
            if (hit) s_list[before + __popc(bm & ((1u << lane) - 1u))] = r;
            if (tid == 0) { int tot = 0; for (int w = 0; w < kBT / 32; ++w) tot += s_warp[w]; s_n = tot; }
            __syncthreads();
        }
        const int nhit = s_n;
        if (nhit > 0) fetch(s_list[0]);
        for (int e = 0; e < nhit; ++e) {
            const int r = s_list[e];
            float* sg = s_g[e & 1];
            Tables& tb = s_tab[e & 1];
            stash(sg);
            if (e + 1 < nhit) fetch(s_list[e + 1]);      // next RoI's gradients are in flight during this one's math
            // ---- per tile row / column: the samples whose taps hit it, in sample order (lo entry before hi entry).
            // Thread (k = tid / 16, q = tid % 16) tests sample q against row / column k; the 16 lanes of a half-warp
            // order their entries with two ballots.
            {
                const BwdMeta m = a.meta[r];
                const int ax = tid >> 8;                             // first 256 threads: rows, the others: columns
                const int k = (tid >> 4) & 15, q = lane & 15, hs = lane & 16;
                {
                    const int ns = 2 * (ax ? c.PW : c.PH);
                    const int coord = (ax ? tx0 : ty0) + k;
                    bool hlo = false, hhi = false;
                    float wl = 0.0f, wh = 0.0f;
                    if (q < ns) {
                        const AxisTap tp = ax ? axis_tap(m.sx, m.bw, q >> 1, q & 1, 2, W) : axis_tap(m.sy, m.bh, q >> 1, q & 1, 2, H);
                        hlo = tp.valid && tp.lo == coord; hhi = tp.valid && tp.hi == coord;
                        wl = tp.h; wh = tp.l;
                    }
                    const unsigned mlo = (__ballot_sync(0xffffffffu, hlo) >> hs) & 0xffffu;
                    const unsigned mhi = (__ballot_sync(0xffffffffu, hhi) >> hs) & 0xffffu;
                    const unsigned below = (1u << q) - 1u;
                    int pos = __popc(mlo & below) + __popc(mhi & below);
                    const int boff = ax ? (q >> 1) * kPitch : (q >> 1) * c.PW * kPitch;
                    if (hlo) {
                        if (ax) { tb.col[k][pos].w = wl; tb.col[k][pos].off = boff; } else { tb.roww[k][pos] = wl; tb.rowb[k][pos] = boff; }
                        ++pos;
                    }
                    if (hhi) {
                        if (ax) { tb.col[k][pos].w = wh; tb.col[k][pos].off = boff; } else { tb.roww[k][pos] = wh; tb.rowb[k][pos] = boff; }
                    }
                    if (q == 0) { if (ax) tb.coln[k] = __popc(mlo) + __popc(mhi); else tb.rown[k] = __popc(mlo) + __popc(mhi); }
                }
            }
            __syncthreads();
            const int nr = tb.rown[row];
            if (nr > 0) {
                const float* gq = sg + cq * 4;
                if (nr <= 4) {                           // the usual case: row terms live in registers
                    float wy[4];
                    const float* gr[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        wy[i] = i < nr ? tb.roww[row][i] : 0.0f;
                        gr[i] = gq + (i < nr ? tb.rowb[row][i] : 0);
                    }
#pragma unroll
                    for (int x = 0; x < kT; ++x) {
                        const int nc = tb.coln[x];
                        for (int j = 0; j < nc; ++j) {
                            const ColTerm ct = tb.col[x][j];
#pragma unroll
                            for (int i = 0; i < 4; ++i) {
                                if (i < nr) {
                                    const float w = wy[i] * ct.w;
                                    const float4 g = *reinterpret_cast<const float4*>(gr[i] + ct.off);
                                    acc[x][0] = fmaf(w, g.x, acc[x][0]); acc[x][1] = fmaf(w, g.y, acc[x][1]);
                                    acc[x][2] = fmaf(w, g.z, acc[x][2]); acc[x][3] = fmaf(w, g.w, acc[x][3]);
                                }
                            }
                        }
                    }
                } else {
#pragma unroll
                    for (int x = 0; x < kT; ++x) {
                        const int nc = tb.coln[x];
                        if (nc == 0) continue;
                        for (int i = 0; i < nr; ++i) {
                            const float wy = tb.roww[row][i];
                            const float* gr = gq + tb.rowb[row][i];
                            for (int j = 0; j < nc; ++j) {
                                const ColTerm ct = tb.col[x][j];
                                const float w = wy * ct.w;
                                const float4 g = *reinterpret_cast<const float4*>(gr + ct.off);
                                acc[x][0] = fmaf(w, g.x, acc[x][0]); acc[x][1] = fmaf(w, g.y, acc[x][1]);
                                acc[x][2] = fmaf(w, g.z, acc[x][2]); acc[x][3] = fmaf(w, g.w, acc[x][3]);
                            }
                        }
                    }
                }
            }
        }
        __syncthreads();                                 // the hit list is rebuilt for the next chunk
    }
    const int y = ty0 + row;
    if (y < H) {
        float* g = a.grad[lvl] + (((long long)img * H + y) * W + tx0) * C + (long long)cg * kCg + cq * 4;
#pragma unroll
        for (int x = 0; x < kT; ++x)
            if (tx0 + x < W) *reinterpret_cast<float4*>(g + (long long)x * C) = make_float4(acc[x][0], acc[x][1], acc[x][2], acc[x][3]);
    }
    __syncthreads();                                     // shared lists / buffers are reused by the next tile
    }
}

}  // namespace

int roi_align_bwd_tile_launch(void* const* grad_feat_ptrs_host, const RoiSets& q, long long R, int B, const b2d_roi_cfg& c,
                              const void* meta, const int* bucket, const int* bcount, const int* guard, cudaStream_t st);

size_t roi_align_bwd_tile_workspace(long long R, int B, int L) {
    const size_t r = (size_t)(R > 0 ? R : 1);
    return r * sizeof(BwdMeta) + 256 + (size_t)B * L * r * 4 + 256 + (size_t)B * L * 4 + 256;
}

// returns 1 if the configuration is not eligible (the caller then uses the generic kernel)
int roi_align_bwd_tile_try(void* const* grad_feat_ptrs_host, const RoiSets& q, const int* levels, long long R, int B,
                           const b2d_roi_cfg& c, void* workspace, cudaStream_t st) {
    if (c.layout != 1 || c.sampling_ratio != 2 || 2 * c.PH > kMaxS || 2 * c.PW > kMaxS || c.PH * c.PW > kMaxBinsT) return 1;
    if (c.C % kCg != 0 || R < 1) return 1;
    for (int l = 0; l < c.num_levels; ++l)
        if (reinterpret_cast<uintptr_t>(grad_feat_ptrs_host[l]) & 15) return 1;
    char* w = (char*)workspace;
    BwdMeta* meta = (BwdMeta*)w; w += ((size_t)R * sizeof(BwdMeta) + 255) & ~(size_t)255;
    int* bucket = (int*)w; w += ((size_t)B * c.num_levels * R * 4 + 255) & ~(size_t)255;
    int* bcount = (int*)w;
    MetaArgs ma;
    memset(&ma, 0, sizeof(ma));
    ma.cfg = c; ma.q = q; ma.levels = levels; ma.R = R;
    k_bwd_meta<<<cdiv(R, 256), 256, 0, st>>>(ma, meta);
    k_bwd_bucket<<<B * c.num_levels, 256, 0, st>>>(meta, R, c.num_levels, bucket, bcount);
    return roi_align_bwd_tile_launch(grad_feat_ptrs_host, q, R, B, c, meta, bucket, bcount, nullptr, st);
}

// the tile kernel alone, on a meta / bucket table that already exists; guard: see TileArgs
int roi_align_bwd_tile_launch(void* const* grad_feat_ptrs_host, const RoiSets& q, long long R, int B, const b2d_roi_cfg& c,
                              const void* meta, const int* bucket, const int* bcount, const int* guard, cudaStream_t st) {
    TileArgs a;
    memset(&a, 0, sizeof(a));
    a.cfg = c;
    int run = 0;
    for (int l = 0; l < c.num_levels; ++l) {
        a.grad[l] = (float*)grad_feat_ptrs_host[l];
        a.tile_off[l] = run;
        a.tiles_x[l] = cdiv(c.W[l], kT);
        run += a.tiles_x[l] * cdiv(c.H[l], kT);
    }
    a.tile_off[c.num_levels] = run;
    a.q = q; a.meta = (const BwdMeta*)meta; a.bucket = bucket; a.bcount = bcount; a.R = R; a.guard = guard;
    a.n_tiles = (unsigned)(run * B);
    unsigned gx = a.n_tiles;
    if (guard) {                                         // persistent: one wave
        int sms = 148, dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        const unsigned wave = (unsigned)cdiv(sms, c.C / kCg);
        if (gx > wave) gx = wave;
    }
    dim3 grid(gx, (unsigned)(c.C / kCg));
    const size_t smem = 2 * sizeof(float) * kMaxBinsT * kPitch + 2 * kTablesBytes;
    B2D_SMEM(k_roi_align_bwd_tile, smem, "k_roi_align_bwd_tile");   // per device
    k_roi_align_bwd_tile<<<grid, kBT, smem, st>>>(a);
    return check_launch("roi_align_bwd(tile)");
}

}  // namespace b2d
