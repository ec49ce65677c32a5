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
#include "nms_common.cuh"

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

// ---- candidate sets past 16384 (cap > kDetT) ------------------------------------------------------------------------
// Round 0 runs b2d_nms on the kDetT best candidates of every image (b2d_topk); an image with at most kDetT candidates is
// then finished.  k_det_continue completes greedy NMS for the others: a candidate is kept iff no KEPT higher-ranked
// candidate suppresses it, so the kept set of a processed prefix is final, and every later candidate a kept one suppresses
// can be dropped (non-kept candidates suppress nothing).  One CTA per image loops: filter the unprocessed candidates against
// the newly kept ones, take the next block of at most kContBlock survivors in rank order, run greedy NMS on it, append its
// survivors -- until max_keep are kept or nothing is left.
constexpr int kDetT = 16384;                  // round-0 candidates per image (the b2d_nms limit)
constexpr int kContThreads = 1024;
constexpr int kContBlock = 1024;              // candidates per continuation round (also the kept-box chunk of the filter)

// round 0: the selected candidates in rank order (b2d_topk output) -> boxes and scores for b2d_nms (presorted)
__global__ void __launch_bounds__(256) k_det_round0(float4* __restrict__ r0_box, float* __restrict__ r0_score,
                                                    const int* __restrict__ r0_idx, const int* __restrict__ r0_n,
                                                    const float4* __restrict__ nms_box, const float* __restrict__ cand_score,
                                                    int cap) {
    const int b = blockIdx.y, r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= r0_n[b]) return;
    const long long i = (long long)b * cap + r0_idx[(long long)b * kDetT + r];
    r0_box[(long long)b * kDetT + r] = nms_box[i];
    r0_score[(long long)b * kDetT + r] = cand_score[i];
}

struct ContArgs {
    const float4* nms_box; const float* cand_score; const int* cand_count;   // [B][cap], [B][cap], [B]
    const int* r0_idx; const int64_t* keep0; const int* keep0_count;          // round 0: [B][kDetT] rank -> candidate, survivors
    int64_t* keep; int* keep_count;                                           // [B][cap] candidate indices, [B]
    uint64_t* list;                                                           // [B][2][cap] unprocessed candidates (ping-pong)
    int* rounds;                                                              // [B] continuation rounds taken
    int cap, max_keep;
    float thr, thr_lo, thr_hi;
};

__device__ __forceinline__ uint64_t cand_comp(const ContArgs& a, long long base, int i) {
    return make_comp(f2key(a.cand_score[base + i]), (uint32_t)i);
}

// block-wide minimum (all threads return it)
__device__ __forceinline__ int block_min(int v, int* s_red) {
    v = __reduce_min_sync(0xffffffffu, v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    int m = s_red[0];
    for (int w = 1; w < kContThreads / 32; ++w) m = min(m, s_red[w]);
    return m;
}

__global__ void __launch_bounds__(kContThreads) k_det_continue(ContArgs a) {
    __shared__ float4 s_box[kContBlock];
    __shared__ float s_area[kContBlock];
    __shared__ uint64_t s_blk[kContBlock];
    __shared__ uint8_t s_dead[kContBlock];
    __shared__ uint32_t s_hist[256];
    __shared__ int s_red[kContThreads / 32];
    __shared__ int s_n, s_m, s_done;
    __shared__ uint64_t s_prefix;
    __shared__ uint32_t s_need;
    const int b = blockIdx.x, tid = threadIdx.x;
    const int count = a.cand_count[b], k0 = a.keep0_count[b];
    const long long base = (long long)b * a.cap;
    int64_t* keep = a.keep + base;
    for (int t = tid; t < k0; t += kContThreads)
        keep[t] = a.r0_idx[(long long)b * kDetT + (int)a.keep0[(long long)b * kDetT + t]];
    if (count <= kDetT || k0 >= a.max_keep) {                        // finished by round 0 (every image, normally)
        if (tid == 0) { a.keep_count[b] = k0; a.rounds[b] = 0; }
        return;
    }
    __syncthreads();                                                 // keep[0, k0) is read back below
    uint64_t* cur = a.list + 2 * base;
    uint64_t* nxt = cur + a.cap;
    // the unprocessed candidates: all below the last one of round 0 (any order: blocks are picked by composite key)
    const uint64_t c_last = cand_comp(a, base, a.r0_idx[(long long)b * kDetT + kDetT - 1]);
    if (tid == 0) s_n = 0;
    __syncthreads();
    for (int i0 = 0; i0 < count; i0 += kContThreads) {
        const int i = i0 + tid;
        const uint64_t c = i < count ? cand_comp(a, base, i) : 0ull;
        const bool in = i < count && c < c_last;
        const int pos = warp_alloc(in, &s_n);
        if (in) cur[pos] = c;
    }
    __syncthreads();
    int n = s_n, kc = k0, filt = 0, rounds = 0;                      // keep[filt, kc): kept, not yet applied to the list
    uint64_t tau = ~0ull;                                            // candidates >= tau are processed
    while (true) {
        // ---- drop the processed candidates and those a kept candidate in keep[filt, kc) suppresses (chunks of kContBlock)
        do {
            __syncthreads();                                         // every thread has read s_m (n) of the previous pass
            const int nk = min(kc - filt, kContBlock);
            for (int t = tid; t < nk; t += kContThreads) {
                const float4 kb = a.nms_box[base + keep[filt + t]];
                s_box[t] = kb; s_area[t] = area_of(kb);
            }
            if (tid == 0) s_m = 0;
            __syncthreads();
            for (int i0 = 0; i0 < n; i0 += kContThreads) {
                const int i = i0 + tid;
                bool live = false;
                uint64_t c = 0ull;
                if (i < n) {
                    c = cur[i];
                    live = c < tau;
                    if (live && nk > 0) {
                        const float4 bx = a.nms_box[base + comp_idx(c)];
                        const float ar = area_of(bx);
                        for (int j = 0; j < nk && live; ++j) live = !suppresses(s_box[j], s_area[j], bx, ar, a.thr, a.thr_lo, a.thr_hi);
                    }
                }
                const int pos = warp_alloc(live, &s_m);
                if (live) nxt[pos] = c;
            }
            __syncthreads();
            n = s_m;
            uint64_t* t = cur; cur = nxt; nxt = t;
            filt += nk;
        } while (filt < kc);
        if (n == 0 || kc >= a.max_keep) break;
        ++rounds;
        // ---- tau = composite of the min(n, kContBlock)-th best remaining candidate (radix select, 8 bits per pass; stops
        // as soon as the remaining count of the current bin is the number still needed)
        const int m = min(n, kContBlock);
        if (tid == 0) { s_prefix = 0ull; s_need = (uint32_t)m; }
        int fixed = 0;                                               // leading bits of tau decided
        while (fixed < 64) {
            const int shift = 56 - fixed;
            for (int t = tid; t < 256; t += kContThreads) s_hist[t] = 0u;
            __syncthreads();
            const uint64_t prefix = s_prefix;
            const uint64_t himask = fixed == 0 ? 0ull : (~0ull << (64 - fixed));
            for (int i0 = 0; i0 < n; i0 += kContThreads) {
                const int i = i0 + tid;
                const uint64_t c = i < n ? cur[i] : 0ull;
                // warp-aggregated: the candidates of a round share their leading bits, so most fall in one bin
                const bool in = i < n && (c & himask) == prefix;
                const uint32_t bin = in ? ((uint32_t)(c >> shift) & 255u) : 256u;
                const unsigned peers = __match_any_sync(0xffffffffu, bin);
                if (in && (tid & 31) == __ffs(peers) - 1) atomicAdd(&s_hist[bin], (uint32_t)__popc(peers));
            }
            __syncthreads();
            if (tid == 0) {
                uint32_t run = 0, need = s_need;
                int d = 255;
                for (; d > 0 && run + s_hist[d] < need; --d) run += s_hist[d];
                s_prefix = prefix | ((uint64_t)d << shift);
                s_need = need - run;
                s_done = (run + s_hist[d] == need) ? 1 : 0;          // the whole bin is taken: tau found
            }
            __syncthreads();
            fixed += 8;
            if (s_done) break;
        }
        tau = s_prefix;                                              // exactly m candidates have composite >= tau
        // ---- the block, in rank order
        if (tid == 0) s_m = 0;
        __syncthreads();
        for (int i0 = 0; i0 < n; i0 += kContThreads) {
            const int i = i0 + tid;
            const bool in = i < n && cur[i] >= tau;
            const int pos = warp_alloc(in, &s_m);
            if (in) s_blk[pos] = cur[i];
        }
        __syncthreads();
        for (int t = m + tid; t < kContBlock; t += kContThreads) s_blk[t] = 0ull;
        bitonic_sort_desc(s_blk, kContBlock);
        for (int t = tid; t < m; t += kContThreads) {
            const float4 bx = a.nms_box[base + comp_idx(s_blk[t])];
            s_box[t] = bx; s_area[t] = area_of(bx); s_dead[t] = 0;
        }
        __syncthreads();
        // ---- greedy NMS on the block; its first candidate survives (no kept candidate suppresses a listed one)
        const int kc0 = kc;
        int r = 0;
        while (r < m && kc < a.max_keep) {
            if (tid == 0) keep[kc] = comp_idx(s_blk[r]);
            ++kc;
            int next = 0x7fffffff;
            for (int t = r + 1 + tid; t < m; t += kContThreads) {
                if (s_dead[t]) continue;
                if (suppresses(s_box[r], s_area[r], s_box[t], s_area[t], a.thr, a.thr_lo, a.thr_hi)) s_dead[t] = 1;
                else next = min(next, t);
            }
            r = block_min(next, s_red);
        }
        filt = kc0;                                                  // the block's survivors filter the rest
        if (kc >= a.max_keep) break;
        __syncthreads();
    }
    if (tid == 0) { a.keep_count[b] = kc; a.rounds[b] = rounds; }
}

}  // namespace b2d

using namespace b2d;

static size_t det_al(size_t v) { return (v + 255) & ~(size_t)255; }

// The workspace of b2d_rcnn_detect / b2d_dense_detect: one carve-up for the launcher, the size query and
// b2d_detect_continuation_rounds (base NULL: sizes only).
struct DetWs {
    float4* cand_box; float4* nms_box; float* cand_score; int* cand_label; int64_t* keep;   // [B][cap]: 48 B per slot
    int* cand_count; uint32_t* maxkey; int* chunk_cnt;
    // cap > kDetT only: round 0 ([B][kDetT]) and the continuation's round counts
    int* r0_idx; int* r0_n; float4* r0_box; float* r0_score; int64_t* keep0; int* keep0_count; int* rounds;
    char* scratch;                // cap <= kDetT: b2d_nms; cap > kDetT: top-k, then b2d_nms, then the continuation lists
    size_t scratch_bytes, total;
};

static DetWs det_layout(char* base, int cap, int B) {
    DetWs d;
    memset(&d, 0, sizeof(d));
    size_t o = 0;
    auto carve = [&](size_t sz) { char* r = base ? base + o : nullptr; o += det_al(sz); return r; };
    const size_t nb = (size_t)B * cap;
    d.cand_box = (float4*)carve(nb * 16);
    d.nms_box = (float4*)carve(nb * 16);
    d.cand_score = (float*)carve(nb * 4);
    d.cand_label = (int*)carve(nb * 4);
    d.keep = (int64_t*)carve(nb * 8);
    d.cand_count = (int*)carve((size_t)B * 4);
    d.maxkey = (uint32_t*)carve((size_t)B * 4);
    d.chunk_cnt = (int*)carve((size_t)B * kDetMaxChunks * 4);
    if (cap <= kDetT) {
        d.scratch_bytes = b2d_nms_workspace_bytes(cap, B);
    } else {
        const size_t nt = (size_t)B * kDetT;
        d.r0_idx = (int*)carve(nt * 4);
        d.r0_n = (int*)carve((size_t)B * 4);
        d.r0_box = (float4*)carve(nt * 16);
        d.r0_score = (float*)carve(nt * 4);
        d.keep0 = (int64_t*)carve(nt * 8);
        d.keep0_count = (int*)carve((size_t)B * 4);
        d.rounds = (int*)carve((size_t)B * 4);
        d.scratch_bytes = std::max(std::max(b2d_topk_workspace_bytes(cap, B, kDetT), b2d_nms_workspace_bytes(kDetT, B)),
                                   nb * 16);                          // lists: 2 x 8 B per slot
    }
    d.scratch = carve(d.scratch_bytes);
    d.total = o;
    return d;
}

// The four stages on a filled DetArgs (everything but the workspace carve-up and the chunking): candidate count,
// candidate write, class-offset boxes, b2d_nms, gather.  events_host (optional, dense form): cudaEvent_t recorded after
// the candidate stage [0] and after the NMS [1].
template <bool kDense>
static int detect_run(DetArgs& p, float* out_box, float* out_score, int64_t* out_label, int* out_count, float* records,
                      float nms_thr_f, int max_per_img, int label_add, int B, int* overflow, void* workspace, size_t ws_bytes,
                      void* const* events_host, cudaStream_t st, const char* what) {
    const int cap = p.cap;
    const DetWs d = det_layout((char*)workspace, cap, B);
    float4* cand_box = d.cand_box;
    float4* nms_box = d.nms_box;
    float* cand_score = d.cand_score;
    int* cand_label = d.cand_label;
    int64_t* keep = d.keep;
    int* cand_count = d.cand_count;
    uint32_t* maxkey = d.maxkey;
    int* chunk_cnt = d.chunk_cnt;
    // chunks of at least 32 rows, at most kDetMaxChunks CTAs per image (8 x 32 CTAs at 1000 proposals, B = 8)
    const long long nmax = p.counts ? p.ld : p.n;
    p.nchunk = (int)std::max(1ll, std::min((long long)kDetMaxChunks, (nmax + 31) / 32));
    p.chunk = (int)std::max(1ll, (nmax + p.nchunk - 1) / p.nchunk);
    p.chunk_cnt = chunk_cnt; p.maxkey = maxkey;
    cudaMemsetAsync(overflow, 0, sizeof(int), st);
    dim3 gc(p.nchunk, B);
    k_rcnn_candidates<false, kDense><<<gc, kDetThreads, 0, st>>>(p, cand_box, cand_score, cand_label, cand_count, overflow);
    k_rcnn_candidates<true, kDense><<<gc, kDetThreads, 0, st>>>(p, cand_box, cand_score, cand_label, cand_count, overflow);
    const int ob = cap <= kDetT ? std::max(1, std::min(16, cdiv(cap, 256))) : std::min(128, cdiv(cap, 256));
    k_rcnn_offset_boxes<<<dim3(ob, B), 256, 0, st>>>(nms_box, cand_box, cand_label, cand_count, maxkey, cap);
    if (int rc = check_launch(what)) return rc;
    if (events_host && events_host[0]) cudaEventRecord((cudaEvent_t)events_host[0], st);
    if (cap <= kDetT) {
        const int rc = b2d_nms(keep, out_count, (const float*)nms_box, cand_score, cap, cand_count, cap, B, nms_thr_f,
                               max_per_img, 0, d.scratch, ws_bytes - (size_t)(d.scratch - (char*)workspace), st);
        if (rc != B2D_OK) return rc;
    } else {
        // round 0 on the kDetT best candidates of every image, then the continuation (see k_det_continue)
        const size_t scratch = ws_bytes - (size_t)(d.scratch - (char*)workspace);
        int rc = b2d_topk(d.r0_idx, d.r0_n, cand_score, cap, cand_count, cap, B, kDetT, d.scratch, scratch, st);
        if (rc != B2D_OK) return rc;
        k_det_round0<<<dim3(kDetT / 256, B), 256, 0, st>>>(d.r0_box, d.r0_score, d.r0_idx, d.r0_n, nms_box, cand_score, cap);
        if ((rc = check_launch(what))) return rc;
        rc = b2d_nms(d.keep0, d.keep0_count, (const float*)d.r0_box, d.r0_score, kDetT, d.r0_n, kDetT, B, nms_thr_f,
                     max_per_img, 1, d.scratch, scratch, st);
        if (rc != B2D_OK) return rc;
        ContArgs a;
        a.nms_box = nms_box; a.cand_score = cand_score; a.cand_count = cand_count;
        a.r0_idx = d.r0_idx; a.keep0 = d.keep0; a.keep0_count = d.keep0_count;
        a.keep = keep; a.keep_count = out_count; a.list = (uint64_t*)d.scratch; a.rounds = d.rounds;
        a.cap = cap; a.max_keep = max_per_img;
        nms_thr_bounds(nms_thr_f, a.thr, a.thr_lo, a.thr_hi);
        k_det_continue<<<B, kContThreads, 0, st>>>(a);
        if ((rc = check_launch(what))) return rc;
    }
    if (events_host && events_host[1]) cudaEventRecord((cudaEvent_t)events_host[1], st);
    dim3 g(cdiv(max_per_img, 256), B);
    k_rcnn_gather<<<g, 256, 0, st>>>(out_box, out_score, out_label, records, keep, out_count, cand_box, cand_score,
                                     cand_label, cap, max_per_img, label_add);
    return check_launch(what);
}

extern "C" {

size_t b2d_rcnn_detect_workspace_bytes(int cap, int B) {
    if (cap < 1 || B < 1 || cap > B2D_DET_MAX_CAP) return 0;
    return det_layout(nullptr, cap, B).total;
}

int b2d_detect_continuation_rounds(int* rounds, const void* workspace, int cap, int B, void* stream) {
    B2D_REQUIRE(rounds && workspace && B >= 1 && cap > kDetT && cap <= B2D_DET_MAX_CAP,
                "detect_continuation_rounds: need a workspace of a call with cap > 16384");
    const DetWs d = det_layout((char*)workspace, cap, B);
    cudaMemcpyAsync(rounds, d.rounds, sizeof(int) * B, cudaMemcpyDeviceToDevice, (cudaStream_t)stream);
    return check_launch("detect_continuation_rounds");
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
    B2D_REQUIRE(cap >= 1 && cap <= B2D_DET_MAX_CAP && max_per_img >= 1 && max_per_img <= std::min(cap, kDetT),
                "rcnn_detect: need 1 <= cap <= 1048576 and max_per_img <= min(cap, 16384)");
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
    B2D_REQUIRE(cap >= 1 && cap <= B2D_DET_MAX_CAP && max_per_img >= 1 && max_per_img <= std::min(cap, kDetT),
                "dense_detect: need 1 <= cap <= 1048576 and max_per_img <= min(cap, 16384)");
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
