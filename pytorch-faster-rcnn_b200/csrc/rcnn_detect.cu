// rcnn_detect.cu -- SURVEY 8(f-3): the RCNN test-time step after RoIAlign / the head convs,
// BBoxHead.predict_bboxes_single_image (lib/heads/bbox_head.py:122-146):
//     score = softmax(cls_out, dim=1)                               [n, C]
//     preds = batched_param2bbox(props, reg_out.t(), means, stds, img_size)   (lib/utils.py:96-106;
//             reg channel = coord * C + class)
//     multiclass_nms(preds.t(), score, range(1, C), nms_iou, min_score, max_per_img, mode)
//             (lib/utils.py:224-269 -> batched_nms :211-221 -> torchvision nms)
// The reference runs ~35 small torch ops and two boolean-mask compactions for this.  Here:
//   k_rcnn_candidates  up to 64 CTAs per image (chunks of consecutive proposals), a warp per proposal, in two
//                      launches: the candidate count of every chunk, then the writes: softmax, candidate test
//                      ('official': every class >= 1 with score >= min_score; 'strict': the arg-max
//                      class only), per-class decode + clamp of the candidates only, ORDERED
//                      compaction (proposal-major, class-minor: the reference's row-major boolean
//                      mask order, which is what breaks score ties in the NMS sort; a chunk starts at
//                      the sum of the earlier chunks' counts) and the maximum coordinate of the
//                      candidate set;
//   k_rcnn_offset_boxes  the class-offset boxes box + fp32(label * max) (lib/utils.py:217-219) for the NMS.
//   b2d_nms (nms.cu)   on the offset boxes, then
//   k_rcnn_gather      the first max_per_img survivors -> un-shifted boxes, scores, labels (and, through
//                      b2d_rcnn_detect_records, the packed all-gather records of dist.pack_detections).
//
// b2d_dense_detect runs the same four stages for the dense one-stage heads (RetinaNet, FCOS / ATSS): utils.multiclass_nms
// (lib/utils.py:224-269) on B images at once.  Its rows are already decoded class-agnostic boxes; each row carries the
// flat anchor / point index it came from, through which k_rcnn_candidates<kDense = true> reads the row's C class values
// in the head's own layout (a per-level table of base pointer, image stride and class stride), applies the score
// transform (none / sigmoid / softmax over C), tests min_score on that raw score and stores score * factor.
#include <algorithm>
#include <cstring>

#include "common.cuh"

namespace b2d {

constexpr int kDetThreads = 256;              // 8 warps: one warp per proposal
constexpr int kDetWarps = kDetThreads / 32;
constexpr int kDetMaxC = 128;                 // classes (incl. background) handled by one warp: 4 per lane
constexpr int kDetMaxChunks = 64;             // CTAs per image; a chunk is at least 32 consecutive proposals

struct DetArgs {
    const float* props; long long ld; const int* counts; long long n;     // [B][4][ld], count per image
    const float* cls; const float* reg; int C, reg_c;                     // cls [B][ld][C]; reg [B][ld][4 * reg_c]
    float ms[8]; int clamp; const float* img_hw;
    float min_score; int strict;
    int cap;                                                              // candidate slots per image
    int chunk, nchunk;                                                    // proposals per CTA, CTAs per image
    int* chunk_cnt;                                                       // [B][kDetMaxChunks] candidates per chunk
    uint32_t* maxkey;                                                     // [B] f2key of the candidate set's max coordinate
    // dense rows (kDense): row i of image b is flat index rows[b][i]; its class c value is
    // lv_base[l][b * lv_img[l] + c * lv_cls[l] + (flat - lv_off[l])] for the level l holding it
    const int* rows;                                                      // [B][ld]
    int nlv, transform;                                                   // transform: 0 none, 1 sigmoid, 2 softmax over C
    long long lv_off[kMaxLevels], lv_img[kMaxLevels], lv_cls[kMaxLevels];
    const float* lv_base[kMaxLevels];
    const float* factor; long long factor_ld;                             // [B][factor_ld] score factor by flat index, or NULL
    unsigned long long chan[2];                                           // bit c: class c is an NMS channel
};

// softmax of proposal i over the C classes (4 classes per lane) and the candidate test
__device__ __forceinline__ void det_row(const DetArgs& p, const float* cls, int i, int lane, float e[4], bool cand[4]) {
    const int C = p.C;
    float x[4];
    float m = -INFINITY;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int c = r * 32 + lane;
        x[r] = c < C ? cls[(long long)i * C + c] : -INFINITY;
        m = fmaxf(m, x[r]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float s = 0.0f;
#pragma unroll
    for (int r = 0; r < 4; ++r) { e[r] = (r * 32 + lane) < C ? expf(x[r] - m) : 0.0f; s += e[r]; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
#pragma unroll
    for (int r = 0; r < 4; ++r) e[r] = e[r] / s;
    if (!p.strict) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int c = r * 32 + lane;
            cand[r] = c >= 1 && c < C && e[r] >= p.min_score;
        }
    } else {
        // arg-max class (first maximum, like torch.max), candidate iff it is a foreground class
        float best = -1.0f;
        int bc = 0x7fffffff;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int c = r * 32 + lane;
            if (c < C && (e[r] > best)) { best = e[r]; bc = c; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ob = __shfl_xor_sync(0xffffffffu, best, o);
            const int oc = __shfl_xor_sync(0xffffffffu, bc, o);
            if (ob > best || (ob == best && oc < bc)) { best = ob; bc = oc; }
        }
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int c = r * 32 + lane;
            cand[r] = c == bc && c >= 1 && best >= p.min_score;
        }
    }
}

// dense row i of image b: its C class values through the level table, the score transform and the candidate test of
// k_mc_candidates (glue.cu): 'official' every NMS channel with score >= min_score; 'strict' the first maximum over ALL
// C channels, a candidate iff it is an NMS channel.  f = the row's score factor (1 without one).
__device__ __forceinline__ void dense_row(const DetArgs& p, int b, int i, int lane, float e[4], bool cand[4], float& f) {
    const int C = p.C;
    const long long fl = p.rows[(long long)b * p.ld + i];
    int l = 0;
    while (l + 1 < p.nlv && fl >= p.lv_off[l + 1]) ++l;
    const float* src = p.lv_base[l] + (long long)b * p.lv_img[l] + (fl - p.lv_off[l]);
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int c = r * 32 + lane;
        e[r] = c < C ? src[(long long)c * p.lv_cls[l]] : -INFINITY;
    }
    if (p.transform == 1) {
#pragma unroll
        for (int r = 0; r < 4; ++r) e[r] = 1.0f / (1.0f + expf(-e[r]));        // torch.sigmoid
    } else if (p.transform == 2) {
        float m = -INFINITY;
#pragma unroll
        for (int r = 0; r < 4; ++r) m = fmaxf(m, e[r]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        float s = 0.0f;
#pragma unroll
        for (int r = 0; r < 4; ++r) { e[r] = (r * 32 + lane) < C ? expf(e[r] - m) : 0.0f; s += e[r]; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
#pragma unroll
        for (int r = 0; r < 4; ++r) e[r] = e[r] / s;
    }
    auto chan = [&](int c) { return ((p.chan[c >> 6] >> (c & 63)) & 1ull) != 0; };
    if (!p.strict) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int c = r * 32 + lane;
            cand[r] = c < C && chan(c) && e[r] >= p.min_score;              // tested on the RAW score (lib/utils.py:248)
        }
    } else {
        float best = -INFINITY;
        int bc = 0x7fffffff;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int c = r * 32 + lane;
            if (c < C && (e[r] > best || bc == 0x7fffffff)) { best = e[r]; bc = c; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ob = __shfl_xor_sync(0xffffffffu, best, o);
            const int oc = __shfl_xor_sync(0xffffffffu, bc, o);
            if (oc != 0x7fffffff && (bc == 0x7fffffff || ob > best || (ob == best && oc < bc))) { best = ob; bc = oc; }
        }
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int c = r * 32 + lane;
            cand[r] = c == bc && c < C && chan(c) && best >= p.min_score;
        }
    }
    f = p.factor ? p.factor[(long long)b * p.factor_ld + fl] : 1.0f;
}

// Grid (nchunk, B): CTA (j, b) takes proposals [j * chunk, (j + 1) * chunk) of image b, a warp per proposal.
//   kWrite == false: the chunk's candidate count -> chunk_cnt[b][j] (and CTA 0 resets maxkey[b]).
//   kWrite == true:  the chunk's candidates are written at (sum of the earlier chunks' counts) + their rank inside
//                    the chunk -- the same proposal-major, class-minor order as one sequential pass -- with the
//                    per-class decode + clamp, and the maximum coordinate of the candidate set goes to maxkey[b];
//                    CTA 0 also stores min(total, cap) and the overflow flag.
//   kDense: rows are dense-head rows (dense_row); the candidate box is the row's box as given, its score score * factor.
template <bool kWrite, bool kDense>
__global__ void __launch_bounds__(kDetThreads) k_rcnn_candidates(DetArgs p, float4* __restrict__ cand_box,
                                                                 float* __restrict__ cand_score,
                                                                 int* __restrict__ cand_label,
                                                                 int* __restrict__ cand_count,
                                                                 int* __restrict__ overflow) {
    __shared__ int s_cnt[kDetWarps], s_off[kDetWarps], s_base;
    const int b = blockIdx.y, j = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = p.counts ? p.counts[b] : (int)p.n;
    const int i_lo = j * p.chunk, i_hi = min(n, i_lo + p.chunk);
    const float* pr = p.props + (long long)b * 4 * p.ld;
    const float* cls = kDense ? nullptr : p.cls + (long long)b * p.ld * p.C;
    const float* reg = kDense ? nullptr : p.reg + (long long)b * p.ld * 4 * p.reg_c;
    const int* ccnt = p.chunk_cnt + (long long)b * kDetMaxChunks;
    float4* cbox = cand_box + (long long)b * p.cap;
    float* cscore = cand_score + (long long)b * p.cap;
    int* clabel = cand_label + (long long)b * p.cap;
    const float img_h = p.clamp ? p.img_hw[2 * b] : 0.0f, img_w = p.clamp ? p.img_hw[2 * b + 1] : 0.0f;
    if (tid == 0) {
        int base = 0, total = 0;
        if (kWrite) {
            for (int q = 0; q < p.nchunk; ++q) {
                if (q == j) base = total;
                total += ccnt[q];
            }
            if (j == 0) {
                cand_count[b] = min(total, p.cap);
                if (total > p.cap) atomicOr(overflow, 1);
            }
        } else if (j == 0) {
            p.maxkey[b] = f2key(-INFINITY);
        }
        s_base = base;
    }
    __syncthreads();
    float vmax = -INFINITY;
    for (int i0 = i_lo; i0 < i_hi; i0 += kDetWarps) {
        const int i = i0 + warp;
        float e[4], f = 1.0f;
        bool cand[4];
        if (i < i_hi) {
            if (kDense) dense_row(p, b, i, lane, e, cand, f);
            else det_row(p, cls, i, lane, e, cand);
        } else {
#pragma unroll
            for (int r = 0; r < 4; ++r) { cand[r] = false; e[r] = 0.0f; }
        }
        unsigned bal[4];
        int ncand = 0;
#pragma unroll
        for (int r = 0; r < 4; ++r) { bal[r] = __ballot_sync(0xffffffffu, cand[r]); ncand += __popc(bal[r]); }
        if (lane == 0) s_cnt[warp] = ncand;
        __syncthreads();
        if (warp == 0) {                                   // exclusive scan of the per-proposal counts of this round
            const int v = lane < kDetWarps ? s_cnt[lane] : 0;
            int incl = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
            }
            if (lane < kDetWarps) s_off[lane] = s_base + incl - v;
            if (lane == kDetWarps - 1) s_cnt[0] = incl;    // round total (s_cnt is dead now)
        }
        __syncthreads();
        if (kWrite && ncand > 0) {
            const Box base{pr[i], pr[p.ld + i], pr[2 * p.ld + i], pr[3 * p.ld + i]};
            int before = s_off[warp];
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                if (cand[r]) {
                    const int c = r * 32 + lane;
                    const int pos = before + __popc(bal[r] & ((1u << lane) - 1u));
                    Box o = base;
                    if (!kDense) {
                        const int rc = p.reg_c > 1 ? c : 0;                 // class-agnostic regression: one box per proposal
                        const float* q = reg + (long long)i * 4 * p.reg_c + rc;
                        o = decode_box(base, q[0], q[p.reg_c], q[2 * p.reg_c], q[3 * p.reg_c], p.ms, p.clamp != 0, img_h,
                                       img_w);
                    }
                    if (pos < p.cap) {
                        cbox[pos] = make_float4(o.x1, o.y1, o.x2, o.y2);
                        cscore[pos] = (kDense && p.factor) ? e[r] * f : e[r];
                        clabel[pos] = c;
                    }
                    vmax = fmaxf(vmax, fmaxf(fmaxf(o.x1, o.y1), fmaxf(o.x2, o.y2)));
                }
                before += __popc(bal[r]);
            }
        }
        __syncthreads();
        if (tid == 0) s_base += s_cnt[0];
        __syncthreads();
    }
    if (kWrite) {
        // bbox.max() over the candidate set (lib/utils.py:217-219): every candidate, also those past the cap
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
        if (lane == 0 && vmax > -INFINITY) atomicMax(&p.maxkey[b], f2key(vmax));
    } else if (tid == 0) {
        p.chunk_cnt[(long long)b * kDetMaxChunks + j] = s_base;
    }
}

// the class-offset boxes box + fp32(label * max) (lib/utils.py:217-219) for the NMS; grid (x, B), grid-stride
__global__ void __launch_bounds__(256) k_rcnn_offset_boxes(float4* __restrict__ nms_box, const float4* __restrict__ cand_box,
                                                           const int* __restrict__ cand_label,
                                                           const int* __restrict__ cand_count,
                                                           const uint32_t* __restrict__ maxkey, int cap) {
    const int b = blockIdx.y;
    const int m = cand_count[b];
    const float mx = key2f(maxkey[b]);
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < m; t += gridDim.x * blockDim.x) {
        const long long k = (long long)b * cap + t;
        const float4 v = cand_box[k];
        const float off = (float)cand_label[k] * mx;           // (label * max_range).to(bbox)
        nms_box[k] = make_float4(v.x + off, v.y + off, v.z + off, v.w + off);
    }
}

// first max_keep survivors (score order) -> [B][4][max_keep] boxes, scores, labels and, if `records` is given, the
// packed rows [B][max_keep][6] = (x1, y1, x2, y2, score, float(label)) of dist.pack_detections (zero past the count).
// label_add is added to the written labels only (a sigmoid dense head's 1-based labels); the NMS offsets used the channel.
__global__ void __launch_bounds__(256) k_rcnn_gather(float* __restrict__ out_box, float* __restrict__ out_score,
                                                     int64_t* __restrict__ out_label, float* __restrict__ records,
                                                     const int64_t* __restrict__ keep,
                                                     const int* __restrict__ keep_count,
                                                     const float4* __restrict__ cand_box,
                                                     const float* __restrict__ cand_score,
                                                     const int* __restrict__ cand_label, int cap, int max_keep,
                                                     int label_add) {
    const int b = blockIdx.y;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= max_keep) return;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    float s = 0.0f;
    int64_t l = 0;
    if (t < keep_count[b]) {
        const long long i = (long long)b * cap + keep[(long long)b * cap + t];
        v = cand_box[i]; s = cand_score[i]; l = (int64_t)cand_label[i] + label_add;
    }
    float* o = out_box + (long long)b * 4 * max_keep;
    o[t] = v.x; o[max_keep + t] = v.y; o[2 * max_keep + t] = v.z; o[3 * max_keep + t] = v.w;
    out_score[(long long)b * max_keep + t] = s;
    out_label[(long long)b * max_keep + t] = l;
    if (records) {
        float* r = records + ((long long)b * max_keep + t) * 6;
        r[0] = v.x; r[1] = v.y; r[2] = v.z; r[3] = v.w; r[4] = s; r[5] = (float)l;
    }
}

}  // namespace b2d

using namespace b2d;

static size_t det_al(size_t v) { return (v + 255) & ~(size_t)255; }

// The four stages on a filled DetArgs (everything but the workspace carve-up and the chunking): candidate count,
// candidate write, class-offset boxes, b2d_nms, gather.  events_host (optional, dense form): cudaEvent_t recorded after
// the candidate stage [0] and after the NMS [1].
template <bool kDense>
static int detect_run(DetArgs& p, float* out_box, float* out_score, int64_t* out_label, int* out_count, float* records,
                      float nms_thr_f, int max_per_img, int label_add, int B, int* overflow, void* workspace, size_t ws_bytes,
                      void* const* events_host, cudaStream_t st, const char* what) {
    const int cap = p.cap;
    char* w = (char*)workspace;
    const size_t nb = (size_t)B * cap;
    float4* cand_box = (float4*)w; w += det_al(nb * 16);
    float4* nms_box = (float4*)w; w += det_al(nb * 16);
    float* cand_score = (float*)w; w += det_al(nb * 4);
    int* cand_label = (int*)w; w += det_al(nb * 4);
    int64_t* keep = (int64_t*)w; w += det_al(nb * 8);
    int* cand_count = (int*)w; w += det_al((size_t)B * 4);
    uint32_t* maxkey = (uint32_t*)w; w += det_al((size_t)B * 4);
    int* chunk_cnt = (int*)w; w += det_al((size_t)B * kDetMaxChunks * 4);
    // chunks of at least 32 rows, at most kDetMaxChunks CTAs per image (8 x 32 CTAs at 1000 proposals, B = 8)
    const long long nmax = p.counts ? p.ld : p.n;
    p.nchunk = (int)std::max(1ll, std::min((long long)kDetMaxChunks, (nmax + 31) / 32));
    p.chunk = (int)std::max(1ll, (nmax + p.nchunk - 1) / p.nchunk);
    p.chunk_cnt = chunk_cnt; p.maxkey = maxkey;
    cudaMemsetAsync(overflow, 0, sizeof(int), st);
    dim3 gc(p.nchunk, B);
    k_rcnn_candidates<false, kDense><<<gc, kDetThreads, 0, st>>>(p, cand_box, cand_score, cand_label, cand_count, overflow);
    k_rcnn_candidates<true, kDense><<<gc, kDetThreads, 0, st>>>(p, cand_box, cand_score, cand_label, cand_count, overflow);
    k_rcnn_offset_boxes<<<dim3(std::max(1, std::min(16, cdiv(cap, 256))), B), 256, 0, st>>>(nms_box, cand_box, cand_label,
                                                                                             cand_count, maxkey, cap);
    if (int rc = check_launch(what)) return rc;
    if (events_host && events_host[0]) cudaEventRecord((cudaEvent_t)events_host[0], st);
    const int rc = b2d_nms(keep, out_count, (const float*)nms_box, cand_score, cap, cand_count, cap, B, nms_thr_f, max_per_img,
                           0, w, ws_bytes - (size_t)(w - (char*)workspace), st);
    if (rc != B2D_OK) return rc;
    if (events_host && events_host[1]) cudaEventRecord((cudaEvent_t)events_host[1], st);
    dim3 g(cdiv(max_per_img, 256), B);
    k_rcnn_gather<<<g, 256, 0, st>>>(out_box, out_score, out_label, records, keep, out_count, cand_box, cand_score,
                                     cand_label, cap, max_per_img, label_add);
    return check_launch(what);
}

extern "C" {

size_t b2d_rcnn_detect_workspace_bytes(int cap, int B) {
    if (cap < 1 || B < 1) return 0;
    const size_t n = (size_t)B * cap;
    return det_al(n * 16) * 2 + det_al(n * 4) * 2 + det_al(n * 8) + det_al((size_t)B * 4) * 2 +
           det_al((size_t)B * kDetMaxChunks * 4) + b2d_nms_workspace_bytes(cap, B);
}

static int rcnn_detect_impl(float* out_box, float* out_score, int64_t* out_label, int* out_count, float* records,
                            const float* props, long long ld, const int* counts, long long n, const float* cls_out,
                            const float* reg_out, int C, int reg_classes, const float* means_host, const float* stds_host,
                            const float* img_hw, float min_score, float nms_thr_f, int max_per_img, int strict, int cap,
                            int B, int* overflow, void* workspace, size_t ws_bytes, void* stream) {
    B2D_REQUIRE(out_box && out_score && out_label && out_count && props && cls_out && reg_out && overflow,
                "rcnn_detect: null pointer");
    B2D_REQUIRE(B >= 1 && n >= 0 && ld >= n && C >= 2 && C <= kDetMaxC && (reg_classes == C || reg_classes == 1),
                "rcnn_detect: need 2 <= C <= 128 and reg_classes in {1, C}");
    B2D_REQUIRE(cap >= 1 && cap <= 16384 && max_per_img >= 1 && max_per_img <= cap, "rcnn_detect: need max_per_img <= cap <= 16384");
    B2D_REQUIRE(workspace && ws_bytes >= b2d_rcnn_detect_workspace_bytes(cap, B), "rcnn_detect: workspace too small");
    DetArgs p;
    memset(&p, 0, sizeof(p));
    p.props = props; p.ld = ld; p.counts = counts; p.n = n;
    p.cls = cls_out; p.reg = reg_out; p.C = C; p.reg_c = reg_classes;
    for (int i = 0; i < 4; ++i) { p.ms[i] = means_host ? means_host[i] : 0.0f; p.ms[4 + i] = stds_host ? stds_host[i] : 1.0f; }
    p.clamp = img_hw ? 1 : 0; p.img_hw = img_hw;
    p.min_score = min_score; p.strict = strict; p.cap = cap;
    return detect_run<false>(p, out_box, out_score, out_label, out_count, records, nms_thr_f, max_per_img, 0, B, overflow,
                             workspace, ws_bytes, nullptr, (cudaStream_t)stream, "rcnn_detect");
}

static int dense_detect_impl(float* out_box, float* out_score, int64_t* out_label, int* out_count, float* records,
                             const float* boxes, long long ld, const int* counts, const int* rows, const b2d_dense_levels* lv_host,
                             int C, int transform, const float* score_factor, long long factor_ld,
                             const unsigned long long* chan_mask_host, float min_score, int label_add, float nms_thr_f,
                             int max_per_img, int strict, int cap, int B, int* overflow, void* workspace, size_t ws_bytes,
                             void* const* events_host, void* stream) {
    B2D_REQUIRE(out_box && out_score && out_label && out_count && boxes && counts && rows && lv_host && chan_mask_host && overflow,
                "dense_detect: null pointer");
    B2D_REQUIRE(B >= 1 && ld >= 1 && C >= 1 && C <= kDetMaxC && transform >= 0 && transform <= 2,
                "dense_detect: need 1 <= C <= 128 and transform in {0, 1, 2}");
    B2D_REQUIRE(cap >= 1 && cap <= 16384 && max_per_img >= 1 && max_per_img <= cap, "dense_detect: need max_per_img <= cap <= 16384");
    B2D_REQUIRE(workspace && ws_bytes >= b2d_rcnn_detect_workspace_bytes(cap, B), "dense_detect: workspace too small");
    const int L = lv_host->num_levels;
    B2D_REQUIRE(L >= 1 && L <= kMaxLevels && lv_host->offset[0] == 0, "dense_detect: need 1..8 levels, the first at offset 0");
    DetArgs p;
    memset(&p, 0, sizeof(p));
    p.props = boxes; p.ld = ld; p.counts = counts; p.n = 0;
    p.C = C; p.min_score = min_score; p.strict = strict; p.cap = cap;
    p.rows = rows; p.nlv = L; p.transform = transform;
    for (int l = 0; l < L; ++l) {
        B2D_REQUIRE(lv_host->base[l] && (l == 0 || lv_host->offset[l] >= lv_host->offset[l - 1]), "dense_detect: bad level table");
        p.lv_off[l] = lv_host->offset[l]; p.lv_base[l] = lv_host->base[l];
        p.lv_img[l] = lv_host->img_stride[l]; p.lv_cls[l] = lv_host->class_stride[l];
    }
    p.factor = score_factor; p.factor_ld = factor_ld;
    p.chan[0] = chan_mask_host[0]; p.chan[1] = chan_mask_host[1];
    return detect_run<true>(p, out_box, out_score, out_label, out_count, records, nms_thr_f, max_per_img, label_add, B, overflow,
                            workspace, ws_bytes, events_host, (cudaStream_t)stream, "dense_detect");
}

int b2d_rcnn_detect(float* out_box, float* out_score, int64_t* out_label, int* out_count, const float* props,
                    long long ld, const int* counts, long long n, const float* cls_out, const float* reg_out, int C,
                    int reg_classes, const float* means_host, const float* stds_host, const float* img_hw,
                    float min_score, float nms_thr_f, int max_per_img, int strict, int cap, int B, int* overflow,
                    void* workspace, size_t ws_bytes, void* stream) {
    return rcnn_detect_impl(out_box, out_score, out_label, out_count, nullptr, props, ld, counts, n, cls_out, reg_out, C,
                            reg_classes, means_host, stds_host, img_hw, min_score, nms_thr_f, max_per_img, strict, cap, B,
                            overflow, workspace, ws_bytes, stream);
}

int b2d_rcnn_detect_records(float* out_box, float* out_score, int64_t* out_label, int* out_count, float* records,
                            const float* props, long long ld, const int* counts, long long n, const float* cls_out,
                            const float* reg_out, int C, int reg_classes, const float* means_host, const float* stds_host,
                            const float* img_hw, float min_score, float nms_thr_f, int max_per_img, int strict, int cap,
                            int B, int* overflow, void* workspace, size_t ws_bytes, void* stream) {
    B2D_REQUIRE(records, "rcnn_detect_records: null records");
    return rcnn_detect_impl(out_box, out_score, out_label, out_count, records, props, ld, counts, n, cls_out, reg_out, C,
                            reg_classes, means_host, stds_host, img_hw, min_score, nms_thr_f, max_per_img, strict, cap, B,
                            overflow, workspace, ws_bytes, stream);
}

int b2d_dense_detect(float* out_box, float* out_score, int64_t* out_label, int* out_count, const float* boxes, long long ld,
                     const int* counts, const int* rows, const b2d_dense_levels* lv_host, int C, int transform,
                     const float* score_factor, long long factor_ld, const unsigned long long* chan_mask_host,
                     float min_score, int label_add, float nms_thr_f, int max_per_img, int strict, int cap, int B,
                     int* overflow, void* workspace, size_t ws_bytes, void* const* events_host, void* stream) {
    return dense_detect_impl(out_box, out_score, out_label, out_count, nullptr, boxes, ld, counts, rows, lv_host, C, transform,
                             score_factor, factor_ld, chan_mask_host, min_score, label_add, nms_thr_f, max_per_img, strict,
                             cap, B, overflow, workspace, ws_bytes, events_host, stream);
}

int b2d_dense_detect_records(float* out_box, float* out_score, int64_t* out_label, int* out_count, float* records,
                             const float* boxes, long long ld, const int* counts, const int* rows,
                             const b2d_dense_levels* lv_host, int C, int transform, const float* score_factor,
                             long long factor_ld, const unsigned long long* chan_mask_host, float min_score, int label_add,
                             float nms_thr_f, int max_per_img, int strict, int cap, int B, int* overflow, void* workspace,
                             size_t ws_bytes, void* const* events_host, void* stream) {
    B2D_REQUIRE(records, "dense_detect_records: null records");
    return dense_detect_impl(out_box, out_score, out_label, out_count, records, boxes, ld, counts, rows, lv_host, C, transform,
                             score_factor, factor_ld, chan_mask_host, min_score, label_add, nms_thr_f, max_per_img, strict,
                             cap, B, overflow, workspace, ws_bytes, events_host, stream);
}

}  // extern "C"
