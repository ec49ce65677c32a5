// select.cu -- K3: fused RPN proposal selection for all (image, level) segments:
//   k_hist      12-bit radix histogram of the monotone logit keys   (multi-block)
//   k_compact   threshold bin from the histogram + candidate compaction (multi-block)
//   k_select    per segment: exact top-k of the candidates by an in-smem linear-key bucket sort (bitonic
//               network / radix narrowing only for heavily tied score maps), anchor generation in
//               registers, delta decode, clip, min-size filter
//   (NMS: nms.cu -- score cut, mask, scan)
//   k_merge_rank  per surviving box: global rank by binary searches over the other levels' lists,
//               scatter to [4, max_num] + sigmoid   (k_merge: single-block form for unsorted lists)
// The launcher runs one chain per FPN level on library-owned streams (see b2d_rpn_proposals).
// Reference: RPNHead.predict_single_image (lib/heads/rpn_head.py:68-120).
//
// Selection and ordering use the *logit* (sigmoid is monotone), ties broken by the
// lowest index; torch.topk's tie order is unspecified (SURVEY 7), so this is the
// documented contract and parity is asserted on tie-free inputs.
#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "pipeline.cuh"
#include "rpn_common.cuh"

namespace b2d {

// ---------------------------------------------------------------- k_hist
// 1024 threads per 16384-element chunk: two rounds of 8 independent loads per thread.  (With 256 threads the chunk
// took 8 dependent DRAM round trips -- 12 us for a kernel that moves 1 MB per image, r1g launch list.)
constexpr int kHcThreads = 1024;

__global__ void __launch_bounds__(kHcThreads) k_hist(RpnLaunch p) {
    __shared__ uint32_t s_h[kHistBins];
    int seg, b, l;
    seg_of(p.lv0, p.lvn, p.L, blockIdx.y, seg, b, l);
    const int n = p.n[l], k = p.kcap[l], nv = seg_valid(p, seg, l);
    if (k >= nv) return;                                 // no selection on this level
    const int start = blockIdx.x * kChunk;
    if (start >= nv) return;
    for (int t = threadIdx.x; t < kHistBins; t += blockDim.x) s_h[t] = 0;
    __syncthreads();
    const float* cls = seg_cls(p, b, l);
    const int end = min(start + kChunk, nv);
    {
        constexpr int kPer = kChunk / kHcThreads;         // 16 independent loads in flight per thread
        float v[kPer];
#pragma unroll
        for (int q = 0; q < kPer; ++q) {
            const int i = start + q * kHcThreads + threadIdx.x;
            v[q] = i < end ? load_logit(cls, n, i, p.score_mode, p.cls_ch) : 0.0f;
        }
#pragma unroll
        for (int q = 0; q < kPer; ++q)
            if (start + q * kHcThreads + (int)threadIdx.x < end) atomicAdd(&s_h[f2key(v[q]) >> (32 - kHistBits)], 1u);
    }
    __syncthreads();
    uint32_t* gh = p.hist + (long long)seg * kHistBins;
    for (int t = threadIdx.x; t < kHistBins; t += blockDim.x)
        if (s_h[t]) atomicAdd(&gh[t], s_h[t]);
}

// Find the largest bin t with sum_{bin >= t} hist[bin] >= k.  blockDim.x == kHcThreads.
__device__ int find_threshold_bin(const uint32_t* __restrict__ gh, int k, uint32_t* s_tmp /*>= 32*/) {
    constexpr int per = kHistBins / kHcThreads, kWarps = kHcThreads / 32;
    uint32_t loc[per];
    uint32_t sum = 0;
#pragma unroll
    for (int q = 0; q < per; ++q) { loc[q] = gh[threadIdx.x * per + q]; sum += loc[q]; }
    // suffix scan over the partial sums: shuffles inside a warp, warp totals through smem
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t v = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_down_sync(0xffffffffu, v, o);
        if (lane + o < 32) v += t;
    }
    __shared__ int s_bin;
    if (lane == 0) s_tmp[warp] = v;
    if (threadIdx.x == 0) s_bin = 0;
    __syncthreads();
    uint32_t above = v - sum;                              // bins owned by higher lanes of this warp
    for (int w = warp + 1; w < kWarps; ++w) above += s_tmp[w];  // ... and by higher warps
    if (above < (uint32_t)k && above + sum >= (uint32_t)k) {
        uint32_t run = above;
        for (int q = per - 1; q >= 0; --q) {
            run += loc[q];
            if (run >= (uint32_t)k) { s_bin = threadIdx.x * per + q; break; }
        }
    }
    __syncthreads();
    return s_bin;
}

// ---------------------------------------------------------------- k_compact
// Two lists per segment: `cand` = keys ABOVE the threshold bin (all of them are selected,
// count < k), `cand2` = keys IN the threshold bin (only the best k - |cand| are).  A block
// stages its candidates (about 1 % of its 16384 elements) in shared memory while it streams
// the chunk with 8 loads in flight per thread and NO barrier in the loop, then leaves with one
// global atomic per list and a coalesced copy (order is irrelevant: they are sorted afterwards).
// Stage overflow (dense candidates: degenerate score maps) appends straight to the global list.
__global__ void __launch_bounds__(kHcThreads) k_compact(RpnLaunch p) {
    constexpr int kCapA = 1536, kCapB = 512;
    __shared__ uint32_t s_tmp[32];
    __shared__ uint64_t s_stageA[kCapA], s_stageB[kCapB];
    __shared__ int s_n, s_n2, s_base, s_base2;
    int seg, b, l;
    seg_of(p.lv0, p.lvn, p.L, blockIdx.y, seg, b, l);
    const int n = p.n[l], k = p.kcap[l], nv = seg_valid(p, seg, l);
    if (k >= nv) return;
    const int start = blockIdx.x * kChunk;
    if (start >= nv) return;
    if (threadIdx.x == 0) { s_n = 0; s_n2 = 0; }
    const float* cls = seg_cls(p, b, l);
    const int end = min(start + kChunk, nv);
    // the whole chunk (16 values per thread) is requested before the threshold search, whose latency it hides
    constexpr int kPer = kChunk / kHcThreads;
    float v[kPer];
#pragma unroll
    for (int q = 0; q < kPer; ++q) {
        const int i = start + q * kHcThreads + threadIdx.x;
        v[q] = i < end ? load_logit(cls, n, i, p.score_mode, p.cls_ch) : 0.0f;
    }
    const int tb = find_threshold_bin(p.hist + (long long)seg * kHistBins, k, s_tmp);   // has barriers
    if (blockIdx.x == 0 && threadIdx.x == 0) p.thr_bin[seg] = tb;
    uint64_t* cand = p.cand + ((long long)b * p.pyr.total + p.pyr.lv[l].offset);
    uint64_t* cand2 = p.cand2 + ((long long)b * p.pyr.total + p.pyr.lv[l].offset);
#pragma unroll
    for (int q = 0; q < kPer; ++q) {
        const int i = start + q * kHcThreads + threadIdx.x;
        const uint32_t key = f2key(v[q]);
        const int bin = (int)(key >> (32 - kHistBits));
        if (i < end && bin > tb) {
            const int pos = atomicAdd(&s_n, 1);
            if (pos < kCapA) s_stageA[pos] = make_comp(key, (uint32_t)i);
            else cand[atomicAdd(&p.cand_count[seg], 1)] = make_comp(key, (uint32_t)i);
        } else if (i < end && bin == tb) {
            const int pos = atomicAdd(&s_n2, 1);
            if (pos < kCapB) s_stageB[pos] = make_comp(key, (uint32_t)i);
            else cand2[atomicAdd(&p.cand2_count[seg], 1)] = make_comp(key, (uint32_t)i);
        }
    }
    __syncthreads();
    const int m = min(s_n, kCapA), m2 = min(s_n2, kCapB);
    if (threadIdx.x == 0 && m > 0) s_base = atomicAdd(&p.cand_count[seg], m);
    if (threadIdx.x == 32 && m2 > 0) s_base2 = atomicAdd(&p.cand2_count[seg], m2);
    __syncthreads();
    for (int t = threadIdx.x; t < m; t += blockDim.x) cand[s_base + t] = s_stageA[t];
    for (int t = threadIdx.x; t < m2; t += blockDim.x) cand2[s_base2 + t] = s_stageB[t];
}

// ---------------------------------------------------------------- k_select
// One block per segment.  Shared memory: kSortCap u64 sort buffer.
__global__ void __launch_bounds__(kSelThreads) k_select(RpnLaunch p) {
    extern __shared__ __align__(16) uint64_t s_buf[];
    __shared__ uint32_t s_h[256];
    __shared__ __align__(16) uint32_t s_off[kHistBins + 4], s_cur[kHistBins], s_wsum[80];
    __shared__ int s_cnt, s_cnt2, s_digit, s_base;
    __shared__ int s_warp[kSelThreads / 32];
    int seg, b, l;
    seg_of(p.lv0, p.lvn, p.L, blockIdx.x, seg, b, l);
    const b2d_level& lv = p.pyr.lv[l];
    const int n = p.n[l], k = p.kcap[l], nv = seg_valid(p, seg, l);
    const float* cls = seg_cls(p, b, l);
    const bool identity = (k >= n) && !p.do_nms;          // AnchorHead path without top-k: keep index order
    int total = 0;
    bool presorted = false;                               // s_buf holds two sorted runs: [0, split_at) and [split_off, ...)
    int split_at = 1 << 30, split_off = 0;
    if (k >= nv) {
        for (int i = threadIdx.x; i < nv; i += blockDim.x)
            s_buf[i] = identity ? make_comp(0xffffffffu, (uint32_t)i)
                                : make_comp(f2key(load_logit(cls, n, i, p.score_mode, p.cls_ch)), (uint32_t)i);
        total = nv;
        if (!identity && nv <= kBucketCap) {
            __syncthreads();
            presorted = bucket_sort_desc(s_buf, s_buf + kBucketCap, total, s_off, s_cur, s_wsum, p.dbg);
        }
    } else {
        uint64_t* listA = p.cand + ((long long)b * p.pyr.total + lv.offset);
        uint64_t* listB = p.cand2 + ((long long)b * p.pyr.total + lv.offset);
        const int sA = p.cand_count[seg];                 // above the threshold bin: all selected (sA < k)
        int m = p.cand2_count[seg];                       // in the threshold bin: best k - sA selected
        int pA = kSelThreads, pB = kSelThreads;
        while (pA < sA) pA <<= 1;
        while (pB < m) pB <<= 1;
        bool done = false;
        if (sA + m <= kBucketCap) {
            for (int i = threadIdx.x; i < sA; i += blockDim.x) s_buf[i] = listA[i];
            for (int i = threadIdx.x; i < m; i += blockDim.x) s_buf[sA + i] = listB[i];
            total = sA + m;
            __syncthreads();
            done = presorted = bucket_sort_desc(s_buf, s_buf + kBucketCap, total, s_off, s_cur, s_wsum, p.dbg);
        }
        if (done) {
        } else if (sA + m <= kSortCap && (sA == 0 || m == 0 || pA + pB > kSortCap)) {
            for (int i = threadIdx.x; i < sA; i += blockDim.x) s_buf[i] = listA[i];
            for (int i = threadIdx.x; i < m; i += blockDim.x) s_buf[sA + i] = listB[i];
            total = sA + m;
        } else if (sA + m <= kSortCap) {
            // Two sorted runs (pow2(sA) + pow2(m) elements) instead of one sort of pow2(sA + m)
            // -- typically 2048 + 1024 instead of 4096 for k = 2000.
            for (int i = threadIdx.x; i < pA; i += blockDim.x) s_buf[i] = i < sA ? listA[i] : 0ull;
            for (int i = threadIdx.x; i < pB; i += blockDim.x) s_buf[pA + i] = i < m ? listB[i] : 0ull;
            __syncthreads();
            bitonic_sort_desc(s_buf, pA);
            bitonic_sort_desc(s_buf + pA, pB);
            split_at = sA; split_off = pA;
            total = sA + m;
            presorted = true;
        } else {
            // radix narrowing of the threshold bin (only reached on heavily tied / degenerate score maps)
            for (int i = threadIdx.x; i < sA; i += blockDim.x) s_buf[i] = listA[i];
            __syncthreads();
            int sel = sA;
            uint64_t* src = listB; uint64_t* dst = listA;   // listA is free once copied
            int shift = 64 - kHistBits - 8;
            while (sel + m > kSortCap) {
                const int bits = shift >= 0 ? 8 : 8 + shift;   // last pass may be narrower
                const int sh = shift >= 0 ? shift : 0;
                const uint32_t dm = (1u << bits) - 1u;
                if (threadIdx.x < 256) s_h[threadIdx.x] = 0;
                __syncthreads();
                for (int i = threadIdx.x; i < m; i += blockDim.x) atomicAdd(&s_h[(uint32_t)(src[i] >> sh) & dm], 1u);
                __syncthreads();
                if (threadIdx.x == 0) {
                    const int need = k - sel;
                    int run = 0, d = (int)dm;
                    for (; d >= 0; --d) { run += (int)s_h[d]; if (run >= need) break; }
                    s_digit = d < 0 ? 0 : d;
                    s_cnt = sel; s_cnt2 = 0;
                }
                __syncthreads();
                const int dg = s_digit;
                for (int i0 = 0; i0 < m; i0 += blockDim.x) {
                    const int i = i0 + threadIdx.x;
                    uint64_t c = 0; int d = -1;
                    if (i < m) { c = src[i]; d = (int)((uint32_t)(c >> sh) & dm); }
                    const int s1 = warp_alloc(d > dg, &s_cnt);
                    if (d > dg) s_buf[s1] = c;
                    const int s2 = warp_alloc(d == dg, &s_cnt2);
                    if (d == dg) dst[s2] = c;
                }
                __syncthreads();
                sel = s_cnt; m = s_cnt2;
                uint64_t* t = src; src = dst; dst = t;
                if (shift <= 0) break;
                shift -= 8;
            }
            for (int i = threadIdx.x; i < m; i += blockDim.x) s_buf[sel + i] = src[i];
            total = sel + m;
        }
    }
    if (!presorted) {
        int p2 = 1;
        while (p2 < total) p2 <<= 1;
        for (int i = total + threadIdx.x; i < p2; i += blockDim.x) s_buf[i] = 0ull;
        __syncthreads();
        bitonic_sort_desc(s_buf, p2);
    }
    const int kk = min(k, total);

    // decode + clip + min-size filter, order preserving
    const float* reg = p.raw ? nullptr : seg_reg(p, b, l);
    const float img_h = p.raw ? 0.0f : p.img_hw[2 * b], img_w = p.raw ? 0.0f : p.img_hw[2 * b + 1];
    const long long so = (long long)b * p.sel_per_img + p.sel_off[l];
    float4* sel_box = p.sel_box + so;
    uint32_t* sel_key = p.sel_key + so;
    int* sel_idx = p.sel_idx + so;
    if (p.raw || !(p.min_size > 0.0f)) {
        // no size filter (min_bbox_size = 0, every reference RPN config): every selected box is kept at its rank, so
        // the order-preserving compaction below (three block barriers per 1024 boxes) is not needed, and the
        // scattered delta loads of a thread's boxes are independent of each other
#pragma unroll 2
        for (int r = threadIdx.x; r < kk; r += blockDim.x) {
            const uint64_t c = s_buf[r < split_at ? r : split_off + (r - split_at)];
            const uint32_t idx = comp_idx(c);
            const uint32_t key = identity ? f2key(load_logit(cls, n, (int)idx, p.score_mode, p.cls_ch)) : comp_key(c);
            Box o{0, 0, 0, 0};
            if (!p.raw) {
                const Box a = anchor_flat(lv, (int)idx);
                o = decode_box(a, reg[idx], reg[n + idx], reg[2 * n + idx], reg[3 * n + idx], p.ms, true, img_h, img_w);
            }
            sel_box[r] = make_float4(o.x1, o.y1, o.x2, o.y2);
            sel_key[r] = key;
            sel_idx[r] = (int)idx;
        }
        if (threadIdx.x == 0) p.sel_count[seg] = kk;
        return;
    }
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    for (int r0 = 0; r0 < kk; r0 += blockDim.x) {
        const int r = r0 + threadIdx.x;
        bool keep = false;
        Box o{0, 0, 0, 0};
        uint32_t key = 0, idx = 0;
        if (r < kk) {
            const uint64_t c = s_buf[r < split_at ? r : split_off + (r - split_at)];
            idx = comp_idx(c);
            key = identity ? f2key(load_logit(cls, n, (int)idx, p.score_mode, p.cls_ch)) : comp_key(c);
            keep = true;
            if (!p.raw) {
                const Box a = anchor_flat(lv, (int)idx);
                o = decode_box(a, reg[idx], reg[n + idx], reg[2 * n + idx], reg[3 * n + idx], p.ms, true, img_h, img_w);
            }
            if (!p.raw && p.min_size > 0.0f)
                keep = ((o.x2 - o.x1) + 1.0f >= p.min_size) && ((o.y2 - o.y1) + 1.0f >= p.min_size);
        }
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        if (lane_id() == 0) s_warp[threadIdx.x >> 5] = __popc(m);
        __syncthreads();
        int before = s_base;
        for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) before += s_warp[w];
        if (keep) {
            const int pos = before + __popc(m & ((1u << lane_id()) - 1u));
            sel_box[pos] = make_float4(o.x1, o.y1, o.x2, o.y2);
            sel_key[pos] = key;
            sel_idx[pos] = (int)idx;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            int t = 0;
            for (int w = 0; w < kSelThreads / 32; ++w) t += s_warp[w];
            s_base += t;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) p.sel_count[seg] = s_base;
}

// ---------------------------------------------------------------- k_merge
// One block per image: gather the per-level NMS survivors (or, without NMS, the
// decoded selections), apply the global top-max_num, write [4, out_ld] + scores.
__global__ void __launch_bounds__(kSelThreads) k_merge(RpnLaunch p, float* __restrict__ props,
                                                       float* __restrict__ scores, int* __restrict__ count,
                                                       int* __restrict__ prov) {
    extern __shared__ __align__(16) uint64_t s_buf[];
    __shared__ int s_off[kMaxLevels + 1];
    const int b = blockIdx.x;
    if (threadIdx.x == 0) {
        int run = 0;
        for (int l = 0; l < p.L; ++l) {
            s_off[l] = run;
            int c = p.do_nms ? p.keep_count[b * p.L + l] : p.sel_count[b * p.L + l];
            if (p.post_nms > 0 && c > p.post_nms) c = p.post_nms;
            run += c;
        }
        s_off[p.L] = run;
    }
    __syncthreads();
    const int total = s_off[p.L];
    const bool topk = (p.max_num > 0) && (total > p.max_num);
    const int nout = topk ? p.max_num : total;
    const float4* m_box = p.do_nms ? p.kept_box : p.sel_box;
    const uint32_t* m_key = p.do_nms ? p.kept_key : p.sel_key;
    const int* m_idx = p.do_nms ? p.kept_idx : p.sel_idx;
    // element t of the level-major concatenation -> (level, position in that level's arrays)
    auto locate = [&](int t, int& l, int& pos) {
        l = 0;
        for (int q = 1; q < p.L; ++q) if (t >= s_off[q]) l = q;
        pos = t - s_off[l];
    };
    // Every level list is already key-descending (NMS keeps score order; the selection is
    // sorted), so the global order is a 5-way merge: the rank of an element is its position
    // in its own level plus, per other level, the number of elements that precede it
    // (binary search; ties go to the earlier concat position).  No sort, two barriers.
    uint32_t* s_key = reinterpret_cast<uint32_t*>(s_buf);
    int* s_rank2t = reinterpret_cast<int*>(s_key + total);
    bool sorted_lists = true;
    for (int l = 0; l < p.L; ++l) if (p.kcap[l] >= p.n[l] && !p.do_nms) sorted_lists = false;
    if (topk && sorted_lists) {
        for (int t = threadIdx.x; t < total; t += blockDim.x) {
            int l, pos; locate(t, l, pos);
            s_key[t] = m_key[(long long)b * p.sel_per_img + p.sel_off[l] + pos];
        }
        __syncthreads();
        for (int t = threadIdx.x; t < total; t += blockDim.x) {
            int l = 0;
            for (int q = 1; q < p.L; ++q) if (t >= s_off[q]) l = q;
            const uint32_t key = s_key[t];
            int rank = t - s_off[l];
            // independent binary searches over the other levels, stepped together for ILP
            int lo[kMaxLevels], hi[kMaxLevels];
#pragma unroll
            for (int q = 0; q < kMaxLevels; ++q) {
                const bool on = q < p.L && q != l;
                lo[q] = on ? s_off[q] : 0; hi[q] = on ? s_off[q + 1] : 0;
            }
            for (int step = 0; step < 15; ++step) {      // 2^14 = kSortCap elements at most
#pragma unroll
                for (int q = 0; q < kMaxLevels; ++q) {
                    if (lo[q] < hi[q]) {
                        const int mid = (lo[q] + hi[q]) >> 1;
                        const uint32_t km = s_key[mid];
                        const bool before = (q < l) ? (km >= key) : (km > key);
                        if (before) lo[q] = mid + 1; else hi[q] = mid;
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < kMaxLevels; ++q)
                if (q < p.L && q != l) rank += lo[q] - s_off[q];
            if (rank < nout) s_rank2t[rank] = t;
        }
        __syncthreads();
    } else if (topk) {
        int p2 = 1;
        while (p2 < total) p2 <<= 1;
        for (int t = threadIdx.x; t < p2; t += blockDim.x) {
            uint64_t c = 0ull;
            if (t < total) {
                int l, pos; locate(t, l, pos);
                c = make_comp(m_key[(long long)b * p.sel_per_img + p.sel_off[l] + pos], (uint32_t)t);
            }
            s_buf[t] = c;
        }
        __syncthreads();
        bitonic_sort_desc(s_buf, p2);
    }
    float* pb = props + (long long)b * 4 * p.out_ld;
    for (int r = threadIdx.x; r < p.out_ld; r += blockDim.x) {
        float4 bx = make_float4(0.f, 0.f, 0.f, 0.f);
        float sc = 0.0f;
        int pv = -1;
        if (r < nout) {
            const int t = !topk ? r : (sorted_lists ? s_rank2t[r] : (int)comp_idx(s_buf[r]));
            int l, pos; locate(t, l, pos);
            const long long o = (long long)b * p.sel_per_img + p.sel_off[l] + pos;
            bx = m_box[o];
            sc = 1.0f / (1.0f + expf(-key2f(m_key[o])));
            pv = (int)(p.pyr.lv[l].offset + m_idx[o]);
        }
        pb[r] = bx.x; pb[p.out_ld + r] = bx.y; pb[2 * p.out_ld + r] = bx.z; pb[3 * p.out_ld + r] = bx.w;
        scores[(long long)b * p.out_ld + r] = sc;
        if (prov) prov[(long long)b * p.out_ld + r] = pv;
        if (p.rec) { float* q = p.rec + ((long long)b * p.out_ld + r) * 5; q[0] = bx.x; q[1] = bx.y; q[2] = bx.z; q[3] = bx.w; q[4] = sc; }
    }
    if (threadIdx.x == 0) count[b] = nout;
}


// ---------------------------------------------------------------- k_merge_rank
// Multi-block form of the merge for the common case (every per-level list is key-descending):
// one thread per surviving element computes its global rank by binary searches over the other
// levels' key lists in global memory (L2-resident) and scatters box/score/provenance straight
// to its output slot.  Replaces a single 1024-thread block per image (69 us, ncu r1d).
__global__ void __launch_bounds__(256) k_merge_rank(RpnLaunch p, float* __restrict__ props,
                                                    float* __restrict__ scores, int* __restrict__ count,
                                                    int* __restrict__ prov) {
    __shared__ int s_off[kMaxLevels + 1];
    const int b = blockIdx.y;
    if (threadIdx.x == 0) {
        int run = 0;
        for (int l = 0; l < p.L; ++l) {
            s_off[l] = run;
            int c = p.do_nms ? p.keep_count[b * p.L + l] : p.sel_count[b * p.L + l];
            if (p.post_nms > 0 && c > p.post_nms) c = p.post_nms;
            run += c;
        }
        s_off[p.L] = run;
    }
    __syncthreads();
    const int total = s_off[p.L];
    const bool topk = (p.max_num > 0) && (total > p.max_num);
    const int nout = topk ? p.max_num : total;
    const float4* m_box = (p.do_nms ? p.kept_box : p.sel_box) + (long long)b * p.sel_per_img;
    const uint32_t* m_key = (p.do_nms ? p.kept_key : p.sel_key) + (long long)b * p.sel_per_img;
    const int* m_idx = (p.do_nms ? p.kept_idx : p.sel_idx) + (long long)b * p.sel_per_img;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    float* pb = props + (long long)b * 4 * p.out_ld;
    if (t == 0) count[b] = nout;
    if (t >= nout && t < p.out_ld) {                     // padding slots
        pb[t] = 0.f; pb[p.out_ld + t] = 0.f; pb[2 * p.out_ld + t] = 0.f; pb[3 * p.out_ld + t] = 0.f;
        scores[(long long)b * p.out_ld + t] = 0.f;
        if (prov) prov[(long long)b * p.out_ld + t] = -1;
        if (p.rec) { float* q = p.rec + ((long long)b * p.out_ld + t) * 5; q[0] = q[1] = q[2] = q[3] = q[4] = 0.f; }
    }
    if (t >= total) return;
    int l = 0;
    for (int q = 1; q < p.L; ++q) if (t >= s_off[q]) l = q;
    const int pos = t - s_off[l];
    const long long o = p.sel_off[l] + pos;
    const uint32_t key = m_key[o];
    int rank = t;
    if (topk) {
        rank = pos;
        int lo[kMaxLevels], hi[kMaxLevels];
#pragma unroll
        for (int q = 0; q < kMaxLevels; ++q) {
            const bool on = q < p.L && q != l;
            lo[q] = 0; hi[q] = on ? s_off[q + 1] - s_off[q] : 0;
        }
        for (int step = 0; step < 15; ++step) {          // 2^14 = kSortCap elements at most
            bool any = false;
#pragma unroll
            for (int q = 0; q < kMaxLevels; ++q) {
                if (lo[q] < hi[q]) {
                    const int mid = (lo[q] + hi[q]) >> 1;
                    const uint32_t km = m_key[p.sel_off[q] + mid];
                    const bool before = (q < l) ? (km >= key) : (km > key);
                    if (before) lo[q] = mid + 1; else hi[q] = mid;
                    any = true;
                }
            }
            if (!any) break;
        }
#pragma unroll
        for (int q = 0; q < kMaxLevels; ++q) rank += lo[q];
    }
    if (rank < nout) {
        const float4 bx = m_box[o];
        pb[rank] = bx.x; pb[p.out_ld + rank] = bx.y; pb[2 * p.out_ld + rank] = bx.z; pb[3 * p.out_ld + rank] = bx.w;
        const float sc = 1.0f / (1.0f + expf(-key2f(key)));
        scores[(long long)b * p.out_ld + rank] = sc;
        if (prov) prov[(long long)b * p.out_ld + rank] = (int)(p.pyr.lv[l].offset + m_idx[o]);
        if (p.rec) { float* q = p.rec + ((long long)b * p.out_ld + rank) * 5; q[0] = bx.x; q[1] = bx.y; q[2] = bx.z; q[3] = bx.w; q[4] = sc; }
    }
}

// ---------------------------------------------------------------- generic segmented top-k
__global__ void __launch_bounds__(kSelThreads) k_topk_small(int* __restrict__ idx, int* __restrict__ out_count,
                                                            const float* __restrict__ values, long long ld,
                                                            const int* __restrict__ counts, long long n, int k) {
    extern __shared__ __align__(16) uint64_t s_buf[];
    const int s = blockIdx.x;
    const int m = counts ? counts[s] : (int)n;
    int p2 = 1;
    while (p2 < m) p2 <<= 1;
    for (int i = threadIdx.x; i < p2; i += blockDim.x)
        s_buf[i] = i < m ? make_comp(f2key(values[(long long)s * ld + i]), (uint32_t)i) : 0ull;
    __syncthreads();
    bitonic_sort_desc(s_buf, p2);
    const int kk = min(k, m);
    for (int r = threadIdx.x; r < k; r += blockDim.x) idx[(long long)s * k + r] = r < kk ? (int)comp_idx(s_buf[r]) : -1;
    if (threadIdx.x == 0) out_count[s] = kk;
}

}  // namespace b2d

using namespace b2d;

namespace b2d {

// Workspace carving shared by the size query and the launcher.
bool rpn_plan(RpnLaunch& p, const b2d_pyramid* pyr, int B, const b2d_rpn_cfg* cfg, char* base, size_t* bytes) {
    memset(&p, 0, sizeof(p));
    p.pyr = *pyr;
    p.B = B; p.L = pyr->num_levels;
    p.lv0 = 0; p.lvn = p.L;
    p.pre_nms = cfg->pre_nms; p.post_nms = cfg->post_nms; p.max_num = cfg->max_num;
    p.score_mode = cfg->score_mode; p.cls_ch = cfg->num_cls_channels > 0 ? cfg->num_cls_channels : 1;
    p.nms_thr = cfg->nms_thr_f; p.min_size = cfg->min_size; p.do_nms = cfg->do_nms;
    p.rec = cfg->records;
    for (int i = 0; i < 4; ++i) { p.ms[i] = cfg->means[i]; p.ms[4 + i] = cfg->stds[i]; }
    long long off = 0;
    int wmax = 0;
    int out_sum = 0;
    for (int l = 0; l < p.L; ++l) {
        const b2d_level& lv = pyr->lv[l];
        const long long n = (long long)lv.A * lv.H * lv.W;
        if (n >= (1ll << 31)) return false;
        p.n[l] = (int)n;
        p.kcap[l] = (cfg->pre_nms > 0 && cfg->pre_nms < n) ? cfg->pre_nms : (int)n;
        if (p.kcap[l] > kSortCap) return false;
        p.sel_off[l] = off;
        off += p.kcap[l];
        const int w = (p.kcap[l] + 63) / 64;
        wmax = w > wmax ? w : wmax;
        p.mask_off[l] = 0;
        out_sum += (cfg->post_nms > 0 && cfg->post_nms < p.kcap[l]) ? cfg->post_nms : p.kcap[l];
    }
    p.sel_per_img = off;
    p.out_ld = cfg->max_num > 0 ? cfg->max_num : out_sum;
    if (cfg->max_num > 0 && out_sum > kSortCap) return false;
    // mask: per segment kcap * ceil(kcap/64) words
    long long moff = 0;
    for (int l = 0; l < p.L; ++l) { p.mask_off[l] = moff; moff += (long long)p.kcap[l] * ((p.kcap[l] + 63) / 64); }
    p.mask_per_img = moff;
    const int S = B * p.L;
    size_t o = 0;
    auto carve = [&](size_t sz) { size_t r = o; o += (sz + 255) & ~(size_t)255; return base ? base + r : (char*)nullptr; };
    p.hist = (uint32_t*)carve((size_t)S * kHistBins * 4);
    p.cand_count = (int*)carve((size_t)S * 4);
    p.cand2_count = (int*)carve((size_t)S * 4);
    p.sel_count = (int*)carve((size_t)S * 4);
    p.keep_count = (int*)carve((size_t)S * 4);
    p.thr_bin = (int*)carve((size_t)S * 4);
    p.n_cut = (int*)carve((size_t)S * 4);
    p.keep1 = (int*)carve((size_t)S * 4);
    p.force_fb = (int*)carve((size_t)B * 4);
    p.nz = (uint32_t*)carve(cfg->do_nms ? (size_t)B * p.sel_per_img * 4 : 0);
    p.zero_bytes = o;                                   // everything above is zeroed per call
    p.cand = (uint64_t*)carve((size_t)B * pyr->total * 8);
    p.cand2 = (uint64_t*)carve((size_t)B * pyr->total * 8);
    p.sel_box = (float4*)carve((size_t)B * p.sel_per_img * 16);
    p.sel_key = (uint32_t*)carve((size_t)B * p.sel_per_img * 4);
    p.sel_idx = (int*)carve((size_t)B * p.sel_per_img * 4);
    const size_t kept = cfg->do_nms ? (size_t)B * p.sel_per_img : 0;
    p.kept_box = (float4*)carve(kept * 16);
    p.kept_key = (uint32_t*)carve(kept * 4);
    p.kept_idx = (int*)carve(kept * 4);
    p.mask = (uint64_t*)carve(cfg->do_nms ? (size_t)B * p.mask_per_img * 8 : 0);
    p.red = (float*)carve((cfg->score_mode == 2 && p.cls_ch > 1) ? (size_t)B * pyr->total * 4 : 0);
    p.dbg_off = o;
    p.dbg_t = (unsigned long long*)carve((size_t)B * kDbgCtas * kDbgStamps * 8);
    *bytes = o;
    return true;
}

// Sigmoid anchor heads with many class channels (RetinaNet: 9 anchors x 80 classes = 64 MB of logits per image): the best
// class logit of every anchor, computed by the whole GPU in one coalesced pass (channel loop per thread, same fmaxf order as
// load_logit mode 2).  The selection kernels then run on the reduced map with score_mode 0 -- inside k_rpn_front the
// 8 CTAs that own an image would pull those 64 MB through 8 SMs (147 us for the stage; 60 us with this pass in front).
__global__ void __launch_bounds__(256) k_class_max(RpnLaunch p, int B) {
    const int l = blockIdx.y;
    const long long n = p.n[l], total = (long long)B * n;
    const float* cls = p.cls[l];
    float* out = p.red + (long long)B * p.pyr.lv[l].offset;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const long long b = t / n, i = t - b * n;
        const float* src = cls + b * n * p.cls_ch + i;
        float m = src[0];
        int c = 1;
        for (; c + 4 <= p.cls_ch; c += 4) {
            const float v0 = src[(long long)c * n], v1 = src[(long long)(c + 1) * n], v2 = src[(long long)(c + 2) * n],
                        v3 = src[(long long)(c + 3) * n];
            m = fmaxf(fmaxf(fmaxf(fmaxf(m, v0), v1), v2), v3);
        }
        for (; c < p.cls_ch; ++c) m = fmaxf(m, src[(long long)c * n]);
        out[t] = m;
    }
}

}  // namespace b2d

namespace {

// Internal per-level streams of b2d_rpn_proposals (created once per device and priority, on the first call; they only ever run
// work that is ordered after / before the caller's stream through the fork / join events).
struct LevelStreams {
    cudaStream_t s[kMaxLevels];
    cudaEvent_t fork, join[kMaxLevels], fork2, join2[kMaxLevels];
    bool ok;
};

// One stream set per (device, priority of the caller's stream): the chains inherit the caller's priority, so two
// concurrent calls on streams of different priority (the staggered image groups of fused.TrainHotPath) neither share
// internal streams nor lose their relative priority.
LevelStreams* level_streams(cudaStream_t caller) {
    constexpr int kPrio = 8;
    static LevelStreams table[64][kPrio];
    static bool made[64][kPrio];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    int lo = 0, hi = 0, pr = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);
    if (cudaStreamGetPriority(caller, &pr) != cudaSuccess) { cudaGetLastError(); pr = lo; }
    int slot = pr - hi;
    slot = slot < 0 ? 0 : (slot >= kPrio ? kPrio - 1 : slot);
    LevelStreams& t = table[dev][slot];
    if (!made[dev][slot]) {
        made[dev][slot] = true;
        t.ok = true;
        for (int l = 0; l < kMaxLevels; ++l) {
            t.ok = t.ok && cudaStreamCreateWithPriority(&t.s[l], cudaStreamNonBlocking, pr) == cudaSuccess;
            t.ok = t.ok && cudaEventCreateWithFlags(&t.join[l], cudaEventDisableTiming) == cudaSuccess;
            t.ok = t.ok && cudaEventCreateWithFlags(&t.join2[l], cudaEventDisableTiming) == cudaSuccess;
        }
        t.ok = t.ok && cudaEventCreateWithFlags(&t.fork, cudaEventDisableTiming) == cudaSuccess;
        t.ok = t.ok && cudaEventCreateWithFlags(&t.fork2, cudaEventDisableTiming) == cudaSuccess;
        if (!t.ok) cudaGetLastError();
    }
    return t.ok ? &t : nullptr;
}

}  // namespace

static thread_local int g_last_launches = 0;

extern "C" {

size_t b2d_rpn_proposals_debug_offset(const b2d_pyramid* pyr_host, int B, const b2d_rpn_cfg* cfg_host) {
    if (!pyr_host || !cfg_host || B < 1) return 0;
    RpnLaunch p;
    size_t bytes = 0;
    if (!rpn_plan(p, pyr_host, B, cfg_host, nullptr, &bytes)) return 0;
    return p.dbg_off;
}

size_t b2d_rpn_proposals_workspace_bytes(const b2d_pyramid* pyr_host, int B, const b2d_rpn_cfg* cfg_host) {
    if (!pyr_host || !cfg_host || B < 1) return 0;
    RpnLaunch p;
    size_t bytes = 0;
    if (!rpn_plan(p, pyr_host, B, cfg_host, nullptr, &bytes)) return 0;
    return bytes;
}

// tg != NULL: the RoI-target stage rides on the proposal kernel when it can (*tg_done = 1), else the caller runs it
static int rpn_proposals_impl(float* props, float* scores, int* count, int* prov, const void* const* cls_ptrs_host,
                              const void* const* reg_ptrs_host, const b2d_pyramid* pyr_host, const float* img_hw, int B,
                              const b2d_rpn_cfg* cfg_host, void* workspace, size_t ws_bytes, const b2d_roi_target_args* tg,
                              int* tg_done, void* stream) {
    B2D_REQUIRE(props && scores && count && cls_ptrs_host && reg_ptrs_host && pyr_host && img_hw && cfg_host,
                "rpn_proposals: null pointer");
    B2D_REQUIRE(B >= 1 && pyr_host->num_levels >= 1 && pyr_host->num_levels <= B2D_MAX_LEVELS,
                "rpn_proposals: bad B / levels");
    RpnLaunch p;
    size_t need = 0;
    B2D_REQUIRE(rpn_plan(p, pyr_host, B, cfg_host, (char*)workspace, &need),
                "rpn_proposals: a level needs a pre-NMS top-k <= 16384 (and the post-NMS concat must fit 16384)");
    B2D_REQUIRE(workspace && ws_bytes >= need, "rpn_proposals: workspace too small");
    for (int l = 0; l < p.L; ++l) { p.cls[l] = (const float*)cls_ptrs_host[l]; p.reg[l] = (const float*)reg_ptrs_host[l]; }
    p.img_hw = img_hw;
    p.dbg = knobs().dbg;
    if (p.dbg != 10) p.dbg_t = nullptr;
    cudaStream_t st = (cudaStream_t)stream;
    int nl = 0;                                           // launches (kernels + memset nodes) of this call
    if (p.score_mode == 2 && p.cls_ch > 1 && p.red) {     // many class channels: reduce once, then select on the reduced map
        int sms = 148, dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        k_class_max<<<dim3(sms * 8, p.L), 256, 0, st>>>(p, B);
        ++nl;
        for (int l = 0; l < p.L; ++l) p.cls[l] = p.red + (long long)B * p.pyr.lv[l].offset;
        p.score_mode = 0; p.cls_ch = 1;
    }
    // function attributes are per device: set on every call (a process may drive several GPUs)
    B2D_SMEM(k_select, kSortCap * 8, "k_select");
    B2D_SMEM(k_merge, kSortCap * 8, "k_merge");
    // Per-level chains.  hist -> compact -> select -> NMS mask -> scan of one level only depends on that level, and
    // all of them but the mask are small latency-bound grids; run as ONE launch per kernel over all levels the step
    // is the sum of the slowest segment of every kernel (166 us at config 2).  Each level therefore gets its own
    // chain on an internal stream (parallel graph branches under capture): the mask work of one level fills the SMs
    // while the other levels sit in their latency-bound kernels.  Joined before the merge.
    int nchains = 1;
    if (knobs().rpn_chains && p.L > 1) nchains = p.L;
    LevelStreams* ls = nchains > 1 ? level_streams(st) : nullptr;
    if (nchains > 1 && !ls) nchains = 1;
    // Score-cut NMS (nms.cu, k_nms_cut): pass 1 on the M = cut * max_num globally best boxes, full pass only for
    // images that need it.  B2D_NMS_CUT = factor (default 1.5), 0 disables.
    int cut_m = 0;
    const bool use_back = rpn_back_applicable(p);        // K4 + merge as one cluster kernel (rpn_back.cu)
    {
        const double f = knobs().nms_cut;
        int kmax = 0;
        long long ksum = 0;
        for (int l = 0; l < p.L; ++l) { kmax = max(kmax, p.kcap[l]); ksum += p.kcap[l]; }
        if (f > 0.0 && p.do_nms && p.max_num > 0 && (nchains > 1 || use_back) && kmax <= 2048 && (double)ksum > f * p.max_num &&
            p.sel_per_img * 4 <= 200 * 1024)
            cut_m = (int)(f * p.max_num);
    }
    // K3 as one cluster kernel (rpn_front.cu) when the plan fits; the per-level chains below otherwise.  The cluster
    // kernels keep their histograms / counters in shared memory and clear what they accumulate into themselves:
    // only the multi-kernel path needs the head of the workspace zeroed.
    bool front_done = false;
    const bool need_zero = !(knobs().rpn_front && !p.raw && use_back && rpn_front_launch_count(p) > 0);
    if (need_zero) { cudaMemsetAsync(workspace, 0, p.zero_bytes, st); ++nl; }
    if (knobs().rpn_front && !p.raw) {
        const int rc = ls ? rpn_front_launch(p, st, ls->s[0], ls->fork, ls->join[0])
                          : rpn_front_launch(p, st, nullptr, nullptr, nullptr);
        if (rc == 1) { front_done = true; nl += rpn_front_launch_count(p); }
        else if (rc != 0) return rc;
    }
    if (!front_done && !need_zero) { cudaMemsetAsync(workspace, 0, p.zero_bytes, st); ++nl; }   // cluster launch unavailable after all
    if (nchains > 1 && !front_done) cudaEventRecord(ls->fork, st);
    for (int c = 0; c < nchains && !front_done; ++c) {
        RpnLaunch q = p;
        cudaStream_t cs = st;
        if (nchains > 1) { q.lv0 = c; q.lvn = 1; cs = ls->s[c]; cudaStreamWaitEvent(cs, ls->fork, 0); }
        const int S = B * q.lvn;
        int max_chunks = 1;
        bool any_select = false;
        for (int l = q.lv0; l < q.lv0 + q.lvn; ++l) {
            if (q.kcap[l] < q.n[l]) { any_select = true; max_chunks = max(max_chunks, cdiv(q.n[l], kChunk)); }
        }
        if (any_select) {
            dim3 grid(max_chunks, S);
            nl += 2;
            k_hist<<<grid, kHcThreads, 0, cs>>>(q);
            if (int rc = check_launch("rpn_proposals/k_hist")) return rc;
            k_compact<<<grid, kHcThreads, 0, cs>>>(q);
            if (int rc = check_launch("rpn_proposals/k_compact")) return rc;
        }
        ++nl;
        k_select<<<S, kSelThreads, kSortCap * 8, cs>>>(q);
        if (int rc = check_launch("rpn_proposals/k_select")) return rc;
        if (q.do_nms && !cut_m && !use_back) {
            int rc = rpn_nms_launch(q, cs);
            if (rc != B2D_OK) return rc;
            nl += 2;
        }
        if (nchains > 1) { cudaEventRecord(ls->join[c], cs); cudaStreamWaitEvent(st, ls->join[c], 0); }
    }
    if (cfg_host->event_after_select) cudaEventRecord((cudaEvent_t)cfg_host->event_after_select, st);
    if (use_back) {
        const bool ride = rpn_back_takes_targets(p, tg);
        const int rc = rpn_back_launch(p, cut_m, props, scores, count, prov, ride ? tg : nullptr, st);
        if (rc == 1) { g_last_launches = nl + 1; if (ride && tg_done) *tg_done = 1; return B2D_OK; }
        return rc == 0 ? B2D_ERR_ARG : rc;
    }
    if (front_done && p.do_nms && !cut_m) {
        if (int rc = rpn_nms_launch(p, st)) return rc;       // plain NMS of all selected boxes, all levels in one launch pair
        nl += 2;
    }
    if (cut_m) {
        if (int rc = rpn_nms_cut_launch(p, cut_m, st)) return rc;
        nl += 1 + 2 + 2;                                     // cut, pass 1 (mask, scan), conditional pass 2 (mask, scan)
        if (knobs().nms_p1_chains == 1) nl += 2 * (nchains - 1);
        // pass 1 on the cut prefixes: one item-walking mask launch + one scan launch over all levels
        // (B2D_NMS_P1_CHAINS=1: the older per-level chains with capacity-sized tile grids, dispatch-bound)
        if (knobs().nms_p1_chains == 1) {
            cudaEventRecord(ls->fork2, st);
            for (int c = 0; c < nchains; ++c) {
                RpnLaunch q = p;
                q.lv0 = c; q.lvn = 1; q.nms_phase = 1;
                cudaStreamWaitEvent(ls->s[c], ls->fork2, 0);
                if (int rc = rpn_nms_launch(q, ls->s[c])) return rc;
                cudaEventRecord(ls->join2[c], ls->s[c]);
                cudaStreamWaitEvent(st, ls->join2[c], 0);
            }
        } else {
            RpnLaunch q = p;
            q.nms_phase = 1;
            if (int rc = rpn_nms_launch(q, st)) return rc;
        }
        RpnLaunch q = p;                                     // pass 2: all levels, skipped per image when pass 1 sufficed
        q.nms_phase = 2;
        if (int rc = rpn_nms_launch(q, st)) return rc;
    }
    bool sorted_lists = true;                            // see k_merge: unsorted only without NMS and without top-k
    int cat = 0;
    for (int l = 0; l < p.L; ++l) {
        if (p.kcap[l] >= p.n[l] && !p.do_nms) sorted_lists = false;
        cat += (p.post_nms > 0 && p.post_nms < p.kcap[l]) ? p.post_nms : p.kcap[l];
    }
    if (sorted_lists) {
        dim3 g(cdiv(max(cat, p.out_ld), 256), B);
        k_merge_rank<<<g, 256, 0, st>>>(p, props, scores, count, prov);
    } else {
        k_merge<<<B, kSelThreads, kSortCap * 8, st>>>(p, props, scores, count, prov);
    }
    g_last_launches = nl + 1;
    return check_launch("rpn_proposals");
}

int b2d_rpn_proposals(float* props, float* scores, int* count, int* prov, const void* const* cls_ptrs_host,
                      const void* const* reg_ptrs_host, const b2d_pyramid* pyr_host, const float* img_hw, int B,
                      const b2d_rpn_cfg* cfg_host, void* workspace, size_t ws_bytes, void* stream) {
    return rpn_proposals_impl(props, scores, count, prov, cls_ptrs_host, reg_ptrs_host, pyr_host, img_hw, B, cfg_host, workspace,
                              ws_bytes, nullptr, nullptr, stream);
}

int b2d_rpn_proposals_targets(float* props, float* scores, int* count, int* prov, const void* const* cls_ptrs_host,
                              const void* const* reg_ptrs_host, const b2d_pyramid* pyr_host, const float* img_hw, int B,
                              const b2d_rpn_cfg* cfg_host, void* workspace, size_t ws_bytes, const b2d_roi_target_args* tg,
                              void* stream) {
    B2D_REQUIRE(tg && tg->labels && tg->max_iou && tg->gt && tg->gt_count && tg->census && tg->chosen && tg->n_chosen,
                "rpn_proposals_targets: null pointer");
    int done = 0;
    const int rc = rpn_proposals_impl(props, scores, count, prov, cls_ptrs_host, reg_ptrs_host, pyr_host, img_hw, B, cfg_host,
                                      workspace, ws_bytes, tg, &done, stream);
    if (rc != B2D_OK || done) return rc;
    RpnLaunch p;
    size_t need = 0;
    if (!rpn_plan(p, pyr_host, B, cfg_host, nullptr, &need)) return B2D_ERR_ARG;
    const int nl = g_last_launches;
    const int rc2 = b2d_roi_targets_fused(tg->labels, tg->max_iou, tg->out_ld, props, p.out_ld, count, p.out_ld, tg->gt, tg->gt_ld,
                                          tg->gt_count, tg->gt_label, B, tg->pos_iou, tg->neg_iou, tg->min_pos_iou, tg->prepend_gt,
                                          tg->census, tg->pos_list, tg->pos_cap, tg->chosen, tg->n_chosen, tg->max_num, tg->pos_num,
                                          tg->seed, tg->seed_step, tg->tar_box, tg->tar_gt, tg->tar_param, tg->tar_label,
                                          tg->tar_is_gt, tg->means, tg->stds, stream);
    g_last_launches = nl + 1;
    return rc2;
}

int b2d_last_launch_count(void) { return g_last_launches; }

static void topk_cfg(long long n, int k, b2d_pyramid& pyr, b2d_rpn_cfg& cfg) {
    memset(&pyr, 0, sizeof(pyr));
    memset(&cfg, 0, sizeof(cfg));
    pyr.num_levels = 1; pyr.total = n;
    pyr.lv[0].H = 1; pyr.lv[0].W = (int)n; pyr.lv[0].A = 1; pyr.lv[0].stride = 1.0f;
    cfg.pre_nms = k; cfg.post_nms = 0; cfg.max_num = 0; cfg.score_mode = 0; cfg.num_cls_channels = 1;
    cfg.do_nms = 0;
    for (int i = 0; i < 4; ++i) cfg.stds[i] = 1.0f;
}

size_t b2d_topk_workspace_bytes(long long n_max, int S, int k) {
    if (n_max <= kSortCap) return 256;
    if (k > kSortCap || n_max >= (1ll << 31)) return 0;
    b2d_pyramid pyr; b2d_rpn_cfg cfg;
    topk_cfg(n_max, k, pyr, cfg);
    RpnLaunch p;
    size_t bytes = 0;
    if (!rpn_plan(p, &pyr, S, &cfg, nullptr, &bytes)) return 0;
    return bytes;
}

namespace b2d {
__global__ void __launch_bounds__(256) k_topk_emit(RpnLaunch p, int* __restrict__ idx, int* __restrict__ out_count, int k) {
    const int s = blockIdx.y;
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    const int c = p.sel_count[s];
    if (r < k) idx[(long long)s * k + r] = r < c ? p.sel_idx[(long long)s * p.sel_per_img + r] : -1;
    if (r == 0) out_count[s] = c;
}
}  // namespace b2d

int b2d_topk(int* idx, int* out_count, const float* values, long long ld, const int* counts, long long n, int S,
             int k, void* workspace, size_t ws_bytes, void* stream) {
    B2D_REQUIRE(idx && out_count && values && S >= 1 && k >= 1, "topk: bad args");
    cudaStream_t st = (cudaStream_t)stream;
    if (n <= kSortCap) {
        B2D_SMEM(k_topk_small, kSortCap * 8, "k_topk_small");   // per device
        k_topk_small<<<S, kSelThreads, kSortCap * 8, st>>>(idx, out_count, values, ld, counts, n, k);
        return check_launch("topk");
    }
    // pyramid-sized inputs: radix histogram + compaction + exact narrowing (the K3 machinery)
    B2D_REQUIRE(ld == n, "topk: n > 16384 needs ld == n");
    B2D_REQUIRE(k <= kSortCap, "topk: k must be <= 16384");
    b2d_pyramid pyr; b2d_rpn_cfg cfg;
    topk_cfg(n, k, pyr, cfg);
    RpnLaunch p;
    size_t need = 0;
    B2D_REQUIRE(rpn_plan(p, &pyr, S, &cfg, (char*)workspace, &need), "topk: unsupported size");
    B2D_REQUIRE(workspace && ws_bytes >= need, "topk: workspace too small");
    p.cls[0] = values; p.reg[0] = nullptr; p.img_hw = nullptr; p.raw = 1; p.seg_n = counts;
    B2D_SMEM(k_select, kSortCap * 8, "k_select");   // per device
    cudaMemsetAsync(workspace, 0, p.zero_bytes, st);
    dim3 grid(cdiv(n, kChunk), S);
    k_hist<<<grid, kHcThreads, 0, st>>>(p);
    k_compact<<<grid, kHcThreads, 0, st>>>(p);
    k_select<<<S, kSelThreads, kSortCap * 8, st>>>(p);
    dim3 g2(cdiv(k, 256), S);
    k_topk_emit<<<g2, 256, 0, st>>>(p, idx, out_count, k);
    return check_launch("topk");
}

}  // extern "C"
