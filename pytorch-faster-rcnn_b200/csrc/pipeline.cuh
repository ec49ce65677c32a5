// pipeline.cuh -- launch descriptor shared by select.cu (K3) and nms.cu (K4) for
// the fused RPN proposal path.
#pragma once
#include "common.cuh"

namespace b2d {

constexpr int kHistBits = 12;
constexpr int kHistBins = 1 << kHistBits;
constexpr int kChunk = 16384;          // elements per block in k_hist / k_compact
constexpr int kSortCap = 16384;        // u64 entries of the in-smem bitonic sort (128 KB)
constexpr int kSelThreads = 1024;

struct RpnLaunch {
    b2d_pyramid pyr;
    const float* cls[kMaxLevels];
    const float* reg[kMaxLevels];
    const float* img_hw;
    int B, L;
    int lv0, lvn;                       // this launch covers levels [lv0, lv0 + lvn) of every image (per-level chains)
    int n[kMaxLevels], kcap[kMaxLevels];
    long long sel_off[kMaxLevels], sel_per_img;
    long long mask_off[kMaxLevels], mask_per_img;
    int pre_nms, post_nms, max_num, score_mode, cls_ch, do_nms, out_ld;
    int raw;                            // 1: plain segmented top-k (no anchors / deltas / decode)
    const int* seg_n;                   // b2d_topk with counts: valid elements per segment, at most n[l] (NULL: n[l])
    int dbg;                            // development knob (B2D_DBG)
    float nms_thr, min_size, ms[8];
    float* rec;                         // optional packed proposal records [B][out_ld][5] (b2d_rpn_cfg::records)
    // workspace
    uint32_t* hist; int* cand_count; int* cand2_count; int* sel_count; int* keep_count; int* thr_bin;
    int* n_cut; int* keep1;             // score-cut NMS: boxes per segment in the first pass, its survivor counts
    int* force_fb;                      // score-cut NMS: per image, 1 = the first pass gave up (sweep kernel), run the full pass
    int nms_phase;                      // 0: plain NMS of all selected boxes; 1: score-cut pass; 2: conditional full pass
    uint32_t* nz;                       // NMS: per selected box, bitmap of its non-zero mask words (nms.cu)
    size_t zero_bytes, dbg_off;
    uint64_t* cand; uint64_t* cand2;
    float* red;                         // score_mode 2 with several class channels: [level][B][n_l] best class logit (k_class_max)
    float4* sel_box; uint32_t* sel_key; int* sel_idx;
    float4* kept_box; uint32_t* kept_key; int* kept_idx;   // NMS survivors, compacted in score order
    uint64_t* mask;
    // development aid (B2D_DBG=10): globaltimer stamps of the cluster kernels, [B][kDbgCtas][kDbgStamps]
    unsigned long long* dbg_t;
};
constexpr int kDbgCtas = 64, kDbgStamps = 16;
__device__ __forceinline__ void dbg_stamp(const RpnLaunch& p, int b, int cta, int k) {
    if (p.dbg_t && threadIdx.x == 0 && cta < kDbgCtas && k < kDbgStamps) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        p.dbg_t[((long long)b * kDbgCtas + cta) * kDbgStamps + k] = t;
    }
}

// elements of segment seg (level l) that take part in the selection
__device__ __forceinline__ int seg_valid(const RpnLaunch& p, int seg, int l) {
    return p.seg_n ? min(max(p.seg_n[seg], 0), p.n[l]) : p.n[l];
}

// launch-local segment index s (b-major over the launch's levels) -> global segment, image, level
__device__ __forceinline__ void seg_of(int lv0, int lvn, int L, int s, int& seg, int& b, int& l) {
    b = s / lvn;
    l = lv0 + (s - b * lvn);
    seg = b * L + l;
}

// rpn_front.cu: cluster kernel for hist + threshold + compact + sort + decode of every segment.
// 1: launched; 0: not applicable (run the multi-kernel path); anything else: error code
int rpn_front_launch(const RpnLaunch& p, cudaStream_t st, cudaStream_t side, cudaEvent_t fork, cudaEvent_t join);
int rpn_front_launch_count(const RpnLaunch& p);      // kernels rpn_front_launch issues for this plan (1 or 2)
// rpn_back.cu: cluster kernel for score cut + sweep mask + scan + merge (one cluster per image)
bool rpn_back_applicable(const RpnLaunch& p);
int rpn_back_launch(const RpnLaunch& p, int cut_m, float* props, float* scores, int* count, int* prov,
                    const ::b2d_roi_target_args* tg, cudaStream_t st);
bool rpn_back_takes_targets(const RpnLaunch& p, const ::b2d_roi_target_args* tg);
// nms.cu: suppression mask + scan over the sel_* arrays of the launch's segments
int rpn_nms_launch(const RpnLaunch& p, cudaStream_t st);
// nms.cu: per image the key of the M-th best selected box over all levels -> n_cut[segment]
int rpn_nms_cut_launch(const RpnLaunch& p, int M, cudaStream_t st);
// nms.cu: pass 1 of the score-cut scheme uses the sweep kernel -> the mask must be zero when it starts
bool rpn_nms_sweep_active(const RpnLaunch& p);

}  // namespace b2d
