// heads.cu -- the head-side glue rows of SURVEY 8(a):
//   a17  BBoxHead.refine_bboxes_single_image (lib/heads/bbox_head.py:100-120): per-class delta
//        pick, GT-column drop (order-preserving compaction), decode + clamp -- one launch/batch
//   a18  ATSS target assignment (K9; lib/heads/fcos_head.py:106-116, 283-368): per (image, GT)
//        the topk nearest cells per level, IoU statistics, then per cell the qualifying GT with the
//        largest IoU (ties -> largest GT index == the reference's sequential `>=` update)
//   a19  FCOS box decode (lib/heads/fcos_head.py:63-75, 578-601): ltrb -> xyxy, clamp,
//        strict min-size test, selection key max_c sigmoid(cls) [* sigmoid(ctr)]
// All of it is small, latency-bound work; the point of the kernels is to replace the
// reference's Python double loops (GT x level, ~40 launches each) by 2-3 launches per batch.
#include <algorithm>
#include <cstring>

#include "common.cuh"

namespace b2d {

// ------------------------------------------------------------------ a17 (+ its test-time form, arg-max labels)
struct RefineArgs {
    const float* props; long long ld; const int* counts; long long n;
    const int64_t* label; const float* reg; int C; const int64_t* is_gt;
    const float* cls; int NC;                   // kArgmax: raw logits [B][ld][NC], label = first maximal index
    float ms[8]; int clamp; const float* img_hw;
};

// kArgmax == false: labels from p.label (the training stages' sampled labels), GT columns dropped.
// kArgmax == true: CascadeRCNN.forward_test's `argmax(cls_out)` (lib/detectors/cascade_rcnn.py:186-190) computed
// in place -- the first maximal index like torch.argmax, background included; nothing is dropped.
template <bool kArgmax>
__global__ void __launch_bounds__(256) k_refine(RefineArgs p, float* __restrict__ out, int* __restrict__ out_count) {
    __shared__ int s_warp[8], s_base;
    const int b = blockIdx.x;
    const int n = p.counts ? p.counts[b] : (int)p.n;
    const float* pr = p.props + (long long)b * 4 * p.ld;
    const int64_t* lab = p.label ? p.label + (long long)b * p.ld : nullptr;
    const int64_t* gtf = p.is_gt ? p.is_gt + (long long)b * p.ld : nullptr;
    const float* reg = p.reg + (long long)b * p.ld * 4 * p.C;
    float* o = out + (long long)b * 4 * p.ld;
    const float img_h = p.clamp ? p.img_hw[2 * b] : 0.0f, img_w = p.clamp ? p.img_hw[2 * b + 1] : 0.0f;
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    for (int i0 = 0; i0 < n; i0 += blockDim.x) {
        const int i = i0 + threadIdx.x;
        const bool keep = i < n && !(!kArgmax && gtf && gtf[i] != 0);
        Box r{0, 0, 0, 0};
        if (keep) {
            const Box base{pr[i], pr[p.ld + i], pr[2 * p.ld + i], pr[3 * p.ld + i]};
            int c = 0;                                                      // reg_out.view(-1, 4, C)[i, :, label]
            if (kArgmax) {
                if (p.C > 1) {
                    const float* x = p.cls + ((long long)b * p.ld + i) * p.NC;
                    float best = x[0];
                    for (int k = 1; k < p.NC; ++k) {
                        const float v = x[k];
                        if (v > best) { best = v; c = k; }
                    }
                }
            } else if (p.C > 1 && lab) {
                c = (int)lab[i];
            }
            const float* q = reg + (long long)i * 4 * p.C + c;
            r = decode_box(base, q[0], q[p.C], q[2 * p.C], q[3 * p.C], p.ms, p.clamp != 0, img_h, img_w);
        }
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        if (lane_id() == 0) s_warp[threadIdx.x >> 5] = __popc(m);
        __syncthreads();
        int before = s_base;
        for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) before += s_warp[w];
        if (keep) {
            const int pos = before + __popc(m & ((1u << lane_id()) - 1u));
            o[pos] = r.x1; o[p.ld + pos] = r.y1; o[2 * p.ld + pos] = r.x2; o[3 * p.ld + pos] = r.y2;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            int t = 0;
            for (int w = 0; w < 8; ++w) t += s_warp[w];
            s_base += t;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) out_count[b] = s_base;
}

// ------------------------------------------------------------------ a18 (K9)
struct AtssArgs {
    b2d_pyramid pyr;                   // A == 1 per level; ws/hs = stride * scale (lib/heads/fcos_head.py:161)
    const float* gt; int gt_ld; const int* gt_count; const int64_t* gt_label;
    const float* img_hw; int topk;
    unsigned long long* key;           // [B][total] winner key: iou bits << 32 | (gt index + 1)
    long long total;
};

constexpr int kAtssMaxCand = B2D_MAX_LEVELS * 16;

__device__ __forceinline__ void cell_point(const b2d_level& lv, int y, int x, float& px, float& py) {
    // bbox2ltrb (lib/heads/fcos_head.py:78-87): full_idx * stride + stride / 2.0
    px = (float)x * lv.stride + lv.stride / 2.0f;
    py = (float)y * lv.stride + lv.stride / 2.0f;
}

// one block per (GT j, image b)
__global__ void __launch_bounds__(256) k_atss_candidates(AtssArgs p) {
    __shared__ int s_cell[kAtssMaxCand];
    __shared__ float s_iou[kAtssMaxCand];
    __shared__ float s_thr;
    const int b = blockIdx.y, j = blockIdx.x;
    const int K = p.gt_count[b];
    if (j >= K) return;
    const float* g = p.gt + (long long)b * 4 * p.gt_ld;
    const Box gb{g[j], g[p.gt_ld + j], g[2 * p.gt_ld + j], g[3 * p.gt_ld + j]};
    const float ga = area_plus1(gb);
    const float gcx = (gb.x2 + gb.x1) / 2.0f, gcy = (gb.y2 + gb.y1) / 2.0f;     // utils.center_of
    // One WARP per level: kk rounds of "smallest (distance, index) strictly above the previous pick" with warp shuffles only.
    // The cells scanned are the 15 x 15 window around the GT centre's cell, not the level: on a square lattice the 9 (topk <=
    // 9) nearest cell centres to a point of the image lie within 4.25 strides of it (a 3 x 3 block next to the nearest cell,
    // grids clipped at the border and both cell-centre conventions included), and a cell 8 or more columns or rows away from
    // floor(centre / stride) -- at most one cell off the nearest -- is at least 6 strides away.  Same picks, same tie order as the
    // full scan (it was 9 block-wide reductions over up to 16 800 cells per level: 220 us for a batch of config 5).
    int ncand = 0;
    {
        const int lane = lane_id(), warp = threadIdx.x >> 5;
        for (int l = 0; l < p.pyr.num_levels; ++l) {
            const b2d_level& lv = p.pyr.lv[l];
            const int n = lv.H * lv.W;
            const int kk = min(p.topk, n);
            if ((l & 7) == warp) {
                int x0 = 0, x1 = lv.W - 1, y0 = 0, y1 = lv.H - 1;
                if (p.topk <= 9 && lv.W >= 3 && lv.H >= 3) {
                    const int cx = min(max((int)floorf(gcx / lv.stride), 0), lv.W - 1);
                    const int cy = min(max((int)floorf(gcy / lv.stride), 0), lv.H - 1);
                    x0 = max(0, cx - 7); x1 = min(lv.W - 1, cx + 7);
                    y0 = max(0, cy - 7); y1 = min(lv.H - 1, cy + 7);
                }
                const int ww = x1 - x0 + 1, wn = ww * (y1 - y0 + 1);
                unsigned long long prev = 0ull;
                for (int r = 0; r < kk; ++r) {
                    unsigned long long best = ~0ull;
                    for (int t = lane; t < wn; t += 32) {
                        const int yy = t / ww, y = y0 + yy, x = x0 + (t - yy * ww);
                        const Box a = anchor_at(lv, 0, y, x);
                        const float dx = (a.x2 + a.x1) / 2.0f - gcx, dy = (a.y2 + a.y1) / 2.0f - gcy;
                        const float d = sqrtf(dx * dx + dy * dy);                      // diff.norm(dim=0)
                        const unsigned long long c = ((unsigned long long)__float_as_uint(d) << 32) | (unsigned)(y * lv.W + x);
                        if ((r == 0 || c > prev) && c < best) best = c;
                    }
                    for (int o = 16; o > 0; o >>= 1) {
                        const unsigned long long t = __shfl_xor_sync(0xffffffffu, best, o);
                        best = t < best ? t : best;
                    }
                    if (lane == 0) {
                        const int i = (int)(best & 0xffffffffu);
                        const int y = i / lv.W, x = i - y * lv.W;
                        const Box a = anchor_at(lv, 0, y, x);
                        s_cell[ncand + r] = (int)lv.offset + i;
                        s_iou[ncand + r] = iou_plus1(a, area_plus1(a), gb, ga);        // utils.calc_iou(close_anchors, gt)
                    }
                    prev = best;
                }
            }
            ncand += kk;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        // mean + unbiased std (lib/heads/fcos_head.py:331-333); accumulated in double, rounded to fp32
        double sum = 0.0;
        for (int c = 0; c < ncand; ++c) sum += (double)s_iou[c];
        const double mean = sum / (double)ncand;
        double var = 0.0;
        for (int c = 0; c < ncand; ++c) { const double d = (double)s_iou[c] - mean; var += d * d; }
        var = ncand > 1 ? var / (double)(ncand - 1) : NAN;
        s_thr = (float)mean + (float)sqrt(var);
    }
    __syncthreads();
    const float thr = s_thr;
    unsigned long long* key = p.key + (long long)b * p.total;
    for (int c = threadIdx.x; c < ncand; c += blockDim.x) {
        const float iou = s_iou[c];
        if (!(iou > thr)) continue;
        const int cell = s_cell[c];
        int l = 0;
        for (int q = 1; q < p.pyr.num_levels; ++q) if (cell >= p.pyr.lv[q].offset) l = q;
        const b2d_level& lv = p.pyr.lv[l];
        const int i = cell - (int)lv.offset;
        const int y = i / lv.W, x = i - y * lv.W;
        float px, py;
        cell_point(lv, y, x, px, py);
        const bool inside = (px - gb.x1 > 0.0f) && (py - gb.y1 > 0.0f) && (gb.x2 - px > 0.0f) && (gb.y2 - py > 0.0f);
        if (!inside) continue;
        // running `iou >= max so far` update in GT order == max over (iou, gt index)
        atomicMax(&key[cell], ((unsigned long long)__float_as_uint(iou) << 32) | (unsigned)(j + 1));
    }
}

__global__ void __launch_bounds__(256) k_atss_finalize(AtssArgs p, int64_t* __restrict__ cls, float* __restrict__ reg,
                                                       float* __restrict__ ctr) {
    const int b = blockIdx.y;
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= p.total) return;
    int l = 0;
    for (int q = 1; q < p.pyr.num_levels; ++q) if (c >= p.pyr.lv[q].offset) l = q;
    const b2d_level& lv = p.pyr.lv[l];
    const int i = (int)(c - lv.offset);
    const int y = i / lv.W, x = i - y * lv.W;
    // paint_value (lib/heads/fcos_head.py:90-94): rows/cols 0..round(img * (1/stride)) inclusive
    const float sc = (float)(1.0 / (double)lv.stride);
    const float img_h = p.img_hw[2 * b], img_w = p.img_hw[2 * b + 1];
    const bool in_img = (float)y <= rintf(img_h * sc) && (float)x <= rintf(img_w * sc);
    int64_t oc = in_img ? 0 : -1;
    float r0 = -1.0f, r1 = -1.0f, r2 = -1.0f, r3 = -1.0f, oct = in_img ? 0.0f : -1.0f;
    const unsigned long long k = p.key[(long long)b * p.total + c];
    if (k != 0ull) {
        const int j = (int)(k & 0xffffffffu) - 1;
        const float* g = p.gt + (long long)b * 4 * p.gt_ld;
        float px, py;
        cell_point(lv, y, x, px, py);
        r0 = px - g[j]; r1 = py - g[p.gt_ld + j]; r2 = g[2 * p.gt_ld + j] - px; r3 = g[3 * p.gt_ld + j] - py;
        oc = p.gt_label[(long long)b * p.gt_ld + j];
        if (oc > 0) {                                                          // centerness (:56-59)
            const float l_ = r0 + 1e-6f, t_ = r1 + 1e-6f, rr = r2 + 1e-6f, bb = r3 + 1e-6f;
            oct = sqrtf((fminf(l_, rr) / fmaxf(l_, rr)) * (fminf(t_, bb) / fmaxf(t_, bb)));
        }
    }
    const long long o = (long long)b * p.total + c;
    cls[o] = oc; ctr[o] = oct;
    reinterpret_cast<float4*>(reg)[o] = make_float4(r0, r1, r2, r3);
}

// ------------------------------------------------------------------ SURVEY 8(f-4): plain FCOS targets
// FCOSHead.single_image_targets (lib/heads/fcos_head.py:371-416): GTs sorted by (+1) area, descending
// (lib/utils.py:362-366), then painted one after the other on every level: a cell takes GT i iff all of
// its ltrb > 0 and thr[level] <= max(ltrb) < thr[level + 1]; later (smaller) GTs overwrite earlier ones.
// Order-free form: per cell the qualifying GT with the SMALLEST area wins (equal areas: the larger
// original index, i.e. the later one of a stable sort; torch.sort leaves ties unspecified).
struct FcosTarArgs {
    b2d_pyramid pyr;
    const float* gt; int gt_ld; const int* gt_count; const int64_t* gt_label;
    const float* img_hw; float thr[kMaxLevels + 1]; long long total;
};

__global__ void __launch_bounds__(256) k_fcos_targets(FcosTarArgs p, int64_t* __restrict__ cls, float* __restrict__ reg,
                                                      float* __restrict__ ctr) {
    const int b = blockIdx.y;
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= p.total) return;
    int l = 0;
    for (int q = 1; q < p.pyr.num_levels; ++q) if (c >= p.pyr.lv[q].offset) l = q;
    const b2d_level& lv = p.pyr.lv[l];
    const int i = (int)(c - lv.offset);
    const int y = i / lv.W, x = i - y * lv.W;
    const float sc = (float)(1.0 / (double)lv.stride);                       // paint_value, as k_atss_finalize
    const float img_h = p.img_hw[2 * b], img_w = p.img_hw[2 * b + 1];
    const bool in_img = (float)y <= rintf(img_h * sc) && (float)x <= rintf(img_w * sc);
    float px, py;
    cell_point(lv, y, x, px, py);
    const float* g = p.gt + (long long)b * 4 * p.gt_ld;
    const int K = p.gt_count[b];
    const float lo = p.thr[l], hi = p.thr[l + 1];
    int win = -1;
    float win_area = 0.0f;
    for (int j = 0; j < K; ++j) {
        const float x1 = g[j], y1 = g[p.gt_ld + j], x2 = g[2 * p.gt_ld + j], y2 = g[3 * p.gt_ld + j];
        const float r0 = px - x1, r1 = py - y1, r2 = x2 - px, r3 = y2 - py;
        const float m = fmaxf(fmaxf(r0, r1), fmaxf(r2, r3));
        const bool ok = r0 > 0.0f && r1 > 0.0f && r2 > 0.0f && r3 > 0.0f && m >= lo && m < hi;
        const float area = ((x2 - x1) + 1.0f) * ((y2 - y1) + 1.0f);
        if (ok && (win < 0 || area <= win_area)) { win = j; win_area = area; }
    }
    int64_t oc = in_img ? 0 : -1;
    float r0 = -1.0f, r1 = -1.0f, r2 = -1.0f, r3 = -1.0f, oct = in_img ? 0.0f : -1.0f;
    if (win >= 0) {
        r0 = px - g[win]; r1 = py - g[p.gt_ld + win]; r2 = g[2 * p.gt_ld + win] - px; r3 = g[3 * p.gt_ld + win] - py;
        oc = p.gt_label[(long long)b * p.gt_ld + win];
        if (oc > 0) {
            const float l_ = r0 + 1e-6f, t_ = r1 + 1e-6f, rr = r2 + 1e-6f, bb = r3 + 1e-6f;
            oct = sqrtf((fminf(l_, rr) / fmaxf(l_, rr)) * (fminf(t_, bb) / fmaxf(t_, bb)));
        }
    }
    const long long o = (long long)b * p.total + c;
    cls[o] = oc; ctr[o] = oct;
    reinterpret_cast<float4*>(reg)[o] = make_float4(r0, r1, r2, r3);
}


// ------------------------------------------------------------------ a19
struct FcosArgs {
    b2d_pyramid pyr;
    const float* cls[kMaxLevels]; const float* reg[kMaxLevels]; const float* ctr[kMaxLevels];
    int C; float reg_mean, reg_std, min_size; const float* img_hw; long long total;
};

// boxes [B][4][total], key [B][total] (= selection score, -inf where the min-size test fails),
// score [B][C][total] = sigmoid(cls), ctrs [B][total] = sigmoid(ctr) (if ctr maps are given)
__global__ void __launch_bounds__(256) k_fcos_decode(FcosArgs p, float* __restrict__ boxes, float* __restrict__ key,
                                                     float* __restrict__ score, float* __restrict__ ctrs) {
    const int b = blockIdx.y;
    const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= p.total) return;
    int l = 0;
    for (int q = 1; q < p.pyr.num_levels; ++q) if (c >= p.pyr.lv[q].offset) l = q;
    const b2d_level& lv = p.pyr.lv[l];
    const long long n = (long long)lv.H * lv.W;
    const int i = (int)(c - lv.offset);
    const int y = i / lv.W, x = i - y * lv.W;
    const float* rg = p.reg[l] + (long long)b * 4 * n;
    float px, py;
    cell_point(lv, y, x, px, py);                                             // ltrb2bbox (:63-75)
    const float l_ = rg[i] * p.reg_std + p.reg_mean, t_ = rg[n + i] * p.reg_std + p.reg_mean;
    const float r_ = rg[2 * n + i] * p.reg_std + p.reg_mean, b_ = rg[3 * n + i] * p.reg_std + p.reg_mean;
    const float mx = p.img_hw[2 * b + 1] - 1.0f, my = p.img_hw[2 * b] - 1.0f;
    const float x1 = fminf(fmaxf(px - l_, 0.0f), mx), y1 = fminf(fmaxf(py - t_, 0.0f), my);
    const float x2 = fminf(fmaxf(r_ + px, 0.0f), mx), y2 = fminf(fmaxf(b_ + py, 0.0f), my);
    float* ob = boxes + (long long)b * 4 * p.total;
    ob[c] = x1; ob[p.total + c] = y1; ob[2 * p.total + c] = x2; ob[3 * p.total + c] = y2;
    const bool ok = ((x2 - x1) + 1.0f > p.min_size) && ((y2 - y1) + 1.0f > p.min_size);   // strict (:602)
    float cs = 1.0f;
    if (p.ctr[l]) {
        cs = 1.0f / (1.0f + expf(-p.ctr[l][(long long)b * n + i]));
        ctrs[(long long)b * p.total + c] = cs;
    }
    float best = -INFINITY;
    for (int k = 0; k < p.C; ++k) {
        const float s = 1.0f / (1.0f + expf(-p.cls[l][((long long)b * p.C + k) * n + i]));
        score[((long long)b * p.C + k) * p.total + c] = s;
        best = fmaxf(best, p.ctr[l] ? s * cs : s);
    }
    key[(long long)b * p.total + c] = ok ? best : -INFINITY;
}

// ------------------------------------------------------------------ a19: batched per-level selection
// FCOSHead.predict_single_image's per-level filter + top-k (lib/heads/fcos_head.py:602-613) for a batch, on the key of
// k_fcos_decode.  Grid (level, image): the CTA counts the valid points (key > -inf) of the earlier levels to find where
// its level starts in the concatenation, then writes either the level's b2d_topk result (more than pre_nms valid
// points) or all its valid points in ascending index order.
constexpr int kDsThreads = 512;
constexpr int kDsSortCap = 16384;             // largest segment b2d_topk sorts at any pitch (one CTA)

struct DsArgs {
    const float* key; long long total; int L, pre; long long P;
    long long off[kMaxLevels]; int n[kMaxLevels];
    const int* topk[kMaxLevels];              // [B][pre] in-level indices, for levels with n > pre; else NULL
    const float* boxes; float* sel_boxes;     // [B][4][total] -> [B][4][P] (optional)
    int* idx; int* count;
};

__device__ __forceinline__ int ds_block_sum(int v, int* s_red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    int t = 0;
#pragma unroll
    for (int w = 0; w < kDsThreads / 32; ++w) t += s_red[w];
    __syncthreads();
    return t;
}

__global__ void __launch_bounds__(kDsThreads) k_dense_select(DsArgs p) {
    __shared__ int s_red[kDsThreads / 32];
    const int l = blockIdx.x, b = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float* key = p.key + (long long)b * p.total;
    auto valid_in = [&](int q) {
        int c = 0;
        for (int i = tid; i < p.n[q]; i += kDsThreads) c += key[p.off[q] + i] > -INFINITY;
        return ds_block_sum(c, s_red);
    };
    auto take = [&](int v) { return (p.pre > 0 && v > p.pre) ? p.pre : v; };
    int base = 0;
    for (int q = 0; q < l; ++q) base += take(valid_in(q));
    const int v = valid_in(l), kl = take(v);
    int* out = p.idx + (long long)b * p.P;
    float* sb = p.sel_boxes ? p.sel_boxes + (long long)b * 4 * p.P : nullptr;
    const float* bx = p.boxes ? p.boxes + (long long)b * 4 * p.total : nullptr;
    auto put = [&](int pos, long long f) {
        out[pos] = (int)f;
        if (sb) { sb[pos] = bx[f]; sb[p.P + pos] = bx[p.total + f]; sb[2 * p.P + pos] = bx[2 * p.total + f]; sb[3 * p.P + pos] = bx[3 * p.total + f]; }
    };
    if (kl < v) {                                                   // top pre_nms by key (region.topk_desc order)
        const int* t = p.topk[l] + (long long)b * p.pre;
        for (int j = tid; j < kl; j += kDsThreads) put(base + j, p.off[l] + t[j]);
    } else {                                                        // every valid point, ascending index
        int run = base;
        for (int i0 = 0; i0 < p.n[l]; i0 += kDsThreads) {
            const int i = i0 + tid;
            const bool ok = i < p.n[l] && key[p.off[l] + i] > -INFINITY;
            const unsigned bal = __ballot_sync(0xffffffffu, ok);
            if (lane == 0) s_red[warp] = __popc(bal);
            __syncthreads();
            int before = 0, total = 0;
#pragma unroll
            for (int w = 0; w < kDsThreads / 32; ++w) { const int c = s_red[w]; before += w < warp ? c : 0; total += c; }
            if (ok) put(run + before + __popc(bal & ((1u << lane) - 1u)), p.off[l] + i);
            run += total;
            __syncthreads();
        }
    }
    if (l == p.L - 1) {                                             // the last level knows the image's count
        const int cnt = base + kl;
        if (tid == 0) p.count[b] = cnt;
        for (long long j = cnt + tid; j < p.P; j += kDsThreads) {
            out[j] = -1;
            if (sb) { sb[j] = 0.0f; sb[p.P + j] = 0.0f; sb[2 * p.P + j] = 0.0f; sb[3 * p.P + j] = 0.0f; }
        }
    }
}

}  // namespace b2d

using namespace b2d;

extern "C" {

int b2d_refine_bboxes(float* out, int* out_count, const float* props, long long ld, const int* counts, long long n,
                      const int64_t* label, const float* reg_out, int C, const int64_t* is_gt,
                      const float* means_host, const float* stds_host, int clamp, const float* img_hw, int B,
                      void* stream) {
    B2D_REQUIRE(out && out_count && props && reg_out && B >= 1 && ld >= 1 && n >= 0 && n <= ld, "refine_bboxes: bad args");
    B2D_REQUIRE(C >= 1 && (C == 1 || label), "refine_bboxes: per-class deltas need labels");
    B2D_REQUIRE(!clamp || img_hw, "refine_bboxes: clamp needs img_hw");
    RefineArgs a;
    memset(&a, 0, sizeof(a));
    a.props = props; a.ld = ld; a.counts = counts; a.n = n; a.label = label; a.reg = reg_out; a.C = C; a.is_gt = is_gt;
    for (int i = 0; i < 4; ++i) { a.ms[i] = means_host ? means_host[i] : 0.0f; a.ms[4 + i] = stds_host ? stds_host[i] : 1.0f; }
    a.clamp = clamp; a.img_hw = img_hw;
    k_refine<false><<<B, 256, 0, (cudaStream_t)stream>>>(a, out, out_count);
    return check_launch("refine_bboxes");
}

int b2d_refine_bboxes_argmax(float* out, int* out_count, const float* props, long long ld, const int* counts, long long n,
                             const float* cls_out, int num_classes, const float* reg_out, int reg_classes,
                             const float* means_host, const float* stds_host, const float* img_hw, int B, void* stream) {
    B2D_REQUIRE(out && out_count && props && cls_out && reg_out && img_hw && B >= 1 && ld >= 1 && n >= 0 && n <= ld,
                "refine_bboxes_argmax: bad args");
    B2D_REQUIRE(num_classes >= 1 && (reg_classes == num_classes || reg_classes == 1),
                "refine_bboxes_argmax: need reg_classes in {1, num_classes}");
    RefineArgs a;
    memset(&a, 0, sizeof(a));
    a.props = props; a.ld = ld; a.counts = counts; a.n = n; a.reg = reg_out; a.C = reg_classes;
    a.cls = cls_out; a.NC = num_classes;
    for (int i = 0; i < 4; ++i) { a.ms[i] = means_host ? means_host[i] : 0.0f; a.ms[4 + i] = stds_host ? stds_host[i] : 1.0f; }
    a.clamp = 1; a.img_hw = img_hw;
    k_refine<true><<<B, 256, 0, (cudaStream_t)stream>>>(a, out, out_count);
    return check_launch("refine_bboxes_argmax");
}

size_t b2d_atss_workspace_bytes(const b2d_pyramid* pyr_host, int B) {
    if (!pyr_host || B < 1) return 0;
    return (size_t)B * (size_t)pyr_host->total * 8;
}

int b2d_atss_assign(int64_t* cls_tar, float* reg_tar, float* ctr_tar, const b2d_pyramid* pyr_host, const float* gt,
                    int gt_ld, const int* gt_count, const int64_t* gt_label, const float* img_hw, int B, int topk,
                    void* workspace, size_t ws_bytes, void* stream) {
    B2D_REQUIRE(cls_tar && reg_tar && ctr_tar && pyr_host && gt && gt_count && gt_label && img_hw, "atss_assign: null pointer");
    B2D_REQUIRE(B >= 1 && gt_ld >= 1 && topk >= 1 && topk <= 16, "atss_assign: need 1 <= topk <= 16");
    B2D_REQUIRE(pyr_host->num_levels >= 1 && pyr_host->num_levels <= B2D_MAX_LEVELS && pyr_host->total < (1ll << 31),
                "atss_assign: bad pyramid");
    for (int l = 0; l < pyr_host->num_levels; ++l)
        B2D_REQUIRE(pyr_host->lv[l].A == 1, "atss_assign: one anchor per cell (lib/heads/fcos_head.py:161)");
    B2D_REQUIRE(workspace && ws_bytes >= b2d_atss_workspace_bytes(pyr_host, B), "atss_assign: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    AtssArgs a;
    a.pyr = *pyr_host; a.gt = gt; a.gt_ld = gt_ld; a.gt_count = gt_count; a.gt_label = gt_label; a.img_hw = img_hw;
    a.topk = topk; a.key = (unsigned long long*)workspace; a.total = pyr_host->total;
    cudaMemsetAsync(workspace, 0, (size_t)B * a.total * 8, st);
    dim3 g1(gt_ld, B);
    k_atss_candidates<<<g1, 256, 0, st>>>(a);
    dim3 g2(cdiv(a.total, 256), B);
    k_atss_finalize<<<g2, 256, 0, st>>>(a, cls_tar, reg_tar, ctr_tar);
    return check_launch("atss_assign");
}

int b2d_fcos_targets(int64_t* cls_tar, float* reg_tar, float* ctr_tar, const b2d_pyramid* pyr_host, const float* gt,
                     int gt_ld, const int* gt_count, const int64_t* gt_label, const float* img_hw,
                     const float* level_thr_host, int B, void* stream) {
    B2D_REQUIRE(cls_tar && reg_tar && ctr_tar && pyr_host && gt && gt_count && gt_label && img_hw && level_thr_host,
                "fcos_targets: null pointer");
    B2D_REQUIRE(B >= 1 && gt_ld >= 1 && pyr_host->num_levels >= 1 && pyr_host->num_levels <= B2D_MAX_LEVELS &&
                pyr_host->total < (1ll << 31), "fcos_targets: bad sizes");
    FcosTarArgs a;
    memset(&a, 0, sizeof(a));
    a.pyr = *pyr_host; a.gt = gt; a.gt_ld = gt_ld; a.gt_count = gt_count; a.gt_label = gt_label; a.img_hw = img_hw;
    a.total = pyr_host->total;
    for (int l = 0; l <= pyr_host->num_levels; ++l) a.thr[l] = level_thr_host[l];
    dim3 g(cdiv(a.total, 256), B);
    k_fcos_targets<<<g, 256, 0, (cudaStream_t)stream>>>(a, cls_tar, reg_tar, ctr_tar);
    return check_launch("fcos_targets");
}

int b2d_fcos_decode(float* boxes, float* key, float* score, float* ctr_score, const void* const* cls_ptrs_host,
                    const void* const* reg_ptrs_host, const void* const* ctr_ptrs_host, const b2d_pyramid* pyr_host,
                    int cls_channels, float reg_mean, float reg_std, float min_size, const float* img_hw, int B,
                    void* stream) {
    B2D_REQUIRE(boxes && key && score && cls_ptrs_host && reg_ptrs_host && pyr_host && img_hw, "fcos_decode: null pointer");
    B2D_REQUIRE(B >= 1 && cls_channels >= 1 && pyr_host->num_levels >= 1 && pyr_host->num_levels <= B2D_MAX_LEVELS,
                "fcos_decode: bad sizes");
    B2D_REQUIRE(!ctr_ptrs_host || ctr_score, "fcos_decode: centerness maps need a ctr_score output");
    FcosArgs a;
    memset(&a, 0, sizeof(a));
    a.pyr = *pyr_host;
    for (int l = 0; l < pyr_host->num_levels; ++l) {
        a.cls[l] = (const float*)cls_ptrs_host[l]; a.reg[l] = (const float*)reg_ptrs_host[l];
        a.ctr[l] = ctr_ptrs_host ? (const float*)ctr_ptrs_host[l] : nullptr;
    }
    a.C = cls_channels; a.reg_mean = reg_mean; a.reg_std = reg_std; a.min_size = min_size; a.img_hw = img_hw;
    a.total = pyr_host->total;
    dim3 g(cdiv(a.total, 256), B);
    k_fcos_decode<<<g, 256, 0, (cudaStream_t)stream>>>(a, boxes, key, score, ctr_score);
    return check_launch("fcos_decode");
}

static size_t ds_al(size_t v) { return (v + 255) & ~(size_t)255; }

// Workspace plan of b2d_dense_select: per level with n > pre_nms a top-k output [B][pre] + counts [B]; one packed key
// buffer [B][n] for the largest such level over kDsSortCap (b2d_topk wants dense segments there); the largest b2d_topk
// workspace.  false: unsupported.
static bool ds_plan(const int* n_host, int L, int B, int pre, size_t* bytes, size_t* topk_at, size_t* packed_at,
                    size_t* ws_at, size_t* ws_len) {
    if (!n_host || L < 1 || L > kMaxLevels || B < 1) return false;
    size_t off = 0, topk_ws = 0;
    long long packed = 0;
    for (int l = 0; l < L; ++l) {
        if (n_host[l] < 0) return false;
        if (topk_at) topk_at[l] = (size_t)-1;
        if (pre > 0 && n_host[l] > pre) {
            if (pre > kDsSortCap) return false;
            const size_t t = b2d_topk_workspace_bytes(n_host[l], B, pre);
            if (t == 0) return false;
            topk_ws = std::max(topk_ws, t);
            if (n_host[l] > kDsSortCap) packed = std::max(packed, (long long)n_host[l]);
            if (topk_at) topk_at[l] = off;
            off += ds_al((size_t)B * pre * 4) + ds_al((size_t)B * 4);
        }
    }
    if (packed_at) *packed_at = off;
    off += ds_al((size_t)B * packed * 4);
    if (ws_at) *ws_at = off;
    if (ws_len) *ws_len = topk_ws;
    *bytes = off + topk_ws + 256;
    return true;
}

size_t b2d_dense_select_workspace_bytes(const int* level_sizes_host, int num_levels, int B, int pre_nms) {
    size_t bytes = 0;
    return ds_plan(level_sizes_host, num_levels, B, pre_nms, &bytes, nullptr, nullptr, nullptr, nullptr) ? bytes : 0;
}

int b2d_dense_select(int* idx, int* count, float* sel_boxes, const float* key, const float* boxes,
                     const int* level_sizes_host, int num_levels, int B, int pre_nms, void* workspace, size_t ws_bytes,
                     void* stream) {
    B2D_REQUIRE(idx && count && key && level_sizes_host && (!sel_boxes || boxes), "dense_select: null pointer");
    size_t bytes = 0, topk_at[kMaxLevels], packed_at = 0, ws_at = 0, ws_len = 0;
    B2D_REQUIRE(ds_plan(level_sizes_host, num_levels, B, pre_nms, &bytes, topk_at, &packed_at, &ws_at, &ws_len),
                "dense_select: unsupported configuration (1..8 levels, a level top-k <= 16384)");
    B2D_REQUIRE(workspace && ws_bytes >= bytes, "dense_select: workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    char* w = (char*)workspace;
    DsArgs a;
    memset(&a, 0, sizeof(a));
    a.key = key; a.L = num_levels; a.pre = pre_nms; a.boxes = boxes; a.sel_boxes = sel_boxes; a.idx = idx; a.count = count;
    long long off = 0, P = 0;
    for (int l = 0; l < num_levels; ++l) {
        const int n = level_sizes_host[l];
        a.off[l] = off; a.n[l] = n;
        P += (pre_nms > 0 && n > pre_nms) ? pre_nms : n;
        off += n;
    }
    a.total = off; a.P = P;
    for (int l = 0; l < num_levels; ++l) {
        if (topk_at[l] == (size_t)-1) continue;
        const int n = a.n[l];
        int* tk = (int*)(w + topk_at[l]);
        int* tc = (int*)(w + topk_at[l] + ds_al((size_t)B * pre_nms * 4));
        const float* v = key + a.off[l];
        long long ld = a.total;
        if (n > kDsSortCap) {                                       // dense [B][n] copy of the level's keys
            float* pk = (float*)(w + packed_at);
            if (cudaMemcpy2DAsync(pk, (size_t)n * 4, v, (size_t)a.total * 4, (size_t)n * 4, B, cudaMemcpyDeviceToDevice, st) !=
                cudaSuccess)
                return check_launch("dense_select(pack)");
            v = pk; ld = n;
        }
        const int rc = b2d_topk(tk, tc, v, ld, nullptr, n, B, pre_nms, w + ws_at, ws_len, st);
        if (rc != B2D_OK) return rc;
        a.topk[l] = tk;
    }
    k_dense_select<<<dim3(num_levels, B), kDsThreads, 0, st>>>(a);
    return check_launch("dense_select");
}

}  // extern "C"
