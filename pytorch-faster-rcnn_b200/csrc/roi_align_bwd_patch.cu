// roi_align_bwd_patch.cu -- K6, patch form ("sorted scatter"): deterministic, atomic-free RoIAlign backward for NHWC fp32
// gradients and 2x2 samples per bin.  Round 2; replaces the tile-gather form (roi_align_bwd_tile.cu, 0.95 ms at config 2:
// ~1100 instructions of loop skeleton per (tile row, RoI) visit and one barrier per visit) where its scratch fits.
//
// The gradient of one RoI is a small dense patch: every cell of the RoI's tap rectangle receives
//     sum_ph sum_pw WY[y][ph] * WX[x][pw] * g[ph][pw] / 4
// with WY[y][ph] = the bilinear row weights of the two samples of bin row ph that land on feature row y (WX likewise):
// the weights of the <= 4 taps of a bin that share a cell are added BEFORE the multiply (2-3 terms per cell instead of
// 6-7 tap terms).  Patches of different RoIs overlap (43 % of the touched cells at config 2), so:
//   k_bwd_meta_mark per-RoI geometry (roi_bwd_common.cuh) and the bitmaps `any` (cell lies in some patch) / `multi` (in two
//                   or more) -- integer atomicOr only, the result does not depend on the order
//   k_bwd_bucket_scan  ascending RoI lists per (image, level); in its last block the exclusive prefix of the patch areas
//                   = scratch slot of every (RoI, cell), raising `fallback` if the patches do not fit the scratch
//   k_bwd_patch     one CTA per (RoI, 128 channels): grad_out[roi] / 4 staged as [bin][channel], the row / column
//                   weight lists built once, then a warp walks its rows of the patch and writes every cell exactly once:
//                   straight into grad_feat if no other patch covers it, else into its scratch slot
//   k_bwd_merge     one CTA per 16 x 16 cell tile: cells in no patch get zeros, cells in several patches the sum of their
//                   scratch slots in ASCENDING RoI order (the sort key of the scatter), cells in one patch are left alone
// Every gradient cell is written once, nothing is zero-filled beforehand, no floating-point atomics: run-to-run
// bit-identical.  Equal to torchvision within rounding (weights are merged per cell), like the tile form.
// Traffic at config 2 (4096 RoIs x 256 channels): 205 MB grad_out + 743 MB of patches (258 MB direct, 485 MB through
// the scratch and back) + 475 MB written by the merge = 1.9 GB.
// If `fallback` is raised the three kernels return at once and the tile kernel (launched behind them, guarded by the
// same flag) does the work: no host synchronisation either way.
#include <cstring>

#include "roi_bwd_common.cuh"

namespace b2d {

int roi_align_bwd_tile_launch(void* const* grad_feat_ptrs_host, const RoiSets& q, long long R, int B, const b2d_roi_cfg& c,
                              const void* meta, const int* bucket, const int* bcount, const int* guard, cudaStream_t st);

namespace {

constexpr int kPT = 128;               // threads per patch CTA: 4 warps, lane = 4 channels
constexpr int kPCg = 128;              // channels per CTA
constexpr int kPPitch = kPCg + 4;      // shared-memory pitch of a bin row (floats)
constexpr int kMaxDim = 32;            // patch rows / columns per block of the weight lists
constexpr int kMaxTerms = 8;           // PH, PW <= 8
constexpr int kMT = 16;                // merge tile side
constexpr int kMThreads = 512;         // merge CTA: warp = tile row
constexpr int kMCap = 512;             // RoIs per bucket chunk

struct __align__(8) Term { float w; int off; };

struct PatchArgs {
    b2d_roi_cfg cfg;
    float* grad[kMaxLevels];
    long long word0[kMaxLevels + 1];   // first bitmap word of each level
    RoiSets q;                         // grad_out rows
    const BwdMeta* meta; const long long* poff;
    unsigned* anyb; unsigned* multi;
    float* scratch; int* flags;        // flags[0] = fallback
    const int* bucket; const int* bcount;
    long long R, cap_cells;
    int tile_off[kMaxLevels + 1], tiles_x[kMaxLevels];
};

// scratch budget: 512 patch cells per RoI on average (config 2: 177; RoIs spread over a level's octave: ~520), at least
// 16 K cells, at most 6 M cells
__host__ __device__ __forceinline__ long long patch_budget_cells(long long R) {
    long long n = R * 512;
    if (n < 16384) n = 16384;
    if (n > 6000000) n = 6000000;
    return n;
}

__device__ __forceinline__ long long patch_area(const BwdMeta& m) {
    return (m.y1 >= m.y0 && m.x1 >= m.x0) ? (long long)(m.y1 - m.y0 + 1) * (m.x1 - m.x0 + 1) : 0;
}

// blocks 0 .. B * L - 1: the ascending RoI list of one (image, level) (k_bwd_bucket with 1024 threads); the last block: the
// exclusive prefix of the patch areas and the fallback flag
__global__ void __launch_bounds__(1024) k_bwd_bucket_scan(const BwdMeta* __restrict__ meta, long long R, int L, int n_maps,
                                                          int* __restrict__ bucket, int* __restrict__ bcount, long long cap_cells,
                                                          long long* __restrict__ poff, int* __restrict__ flags) {
    __shared__ long long s_w[32];
    __shared__ long long s_base;
    if (threadIdx.x == 0) s_base = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if ((int)blockIdx.x < n_maps) {
        const int img = blockIdx.x / L, lvl = blockIdx.x - img * L;
        int* out = bucket + (long long)blockIdx.x * R;
        for (long long r0 = 0; r0 < R; r0 += 1024) {
            const long long r = r0 + threadIdx.x;
            bool hit = false;
            if (r < R) { const int4 h = *reinterpret_cast<const int4*>(meta + r); hit = h.x == img && h.y == lvl; }
            const unsigned bm = __ballot_sync(0xffffffffu, hit);
            if (lane == 0) s_w[warp] = __popc(bm);
            __syncthreads();
            long long before = s_base;
            for (int w = 0; w < warp; ++w) before += s_w[w];
            if (hit) out[before + __popc(bm & ((1u << lane) - 1u))] = (int)r;
            __syncthreads();
            if (threadIdx.x == 0) { long long t = 0; for (int w = 0; w < 32; ++w) t += s_w[w]; s_base += t; }
            __syncthreads();
        }
        if (threadIdx.x == 0) bcount[blockIdx.x] = (int)s_base;
        return;
    }
    int live = 0;                                       // records of RoIs (batched form: slots below their image's count)
    for (long long r0 = 0; r0 < R; r0 += 1024) {
        const long long r = r0 + threadIdx.x;
        long long a = 0;
        if (r < R) { const BwdMeta m = meta[r]; a = patch_area(m); live += m.img >= 0; }
        long long inc = a;
        for (int d = 1; d < 32; d <<= 1) {
            const long long t = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc += t;
        }
        if (lane == 31) s_w[warp] = inc;
        __syncthreads();
        long long before = s_base;
        for (int w = 0; w < warp; ++w) before += s_w[w];
        if (r < R) poff[r] = before + inc - a;
        __syncthreads();
        if (threadIdx.x == 0) { long long t = 0; for (int w = 0; w < 32; ++w) t += s_w[w]; s_base += t; }
        __syncthreads();
    }
    // the budget of the RoIs actually present, so that the batched entry (empty slots included in R) takes the patch or
    // the tile form exactly when the unbatched call on the compacted list does
    live = (int)__reduce_add_sync(0xffffffffu, (unsigned)live);
    if (lane == 0) s_w[warp] = live;
    __syncthreads();
    if (threadIdx.x == 0) {
        long long n = 0;
        for (int w = 0; w < 32; ++w) n += s_w[w];
        poff[R] = s_base;
        flags[0] = s_base > min(cap_cells, patch_budget_cells(n)) ? 1 : 0;
    }
}

// one warp per RoI: its geometry record, then the rows of its patch into the `any` / `multi` bitmaps (lanes over rows)
__global__ void __launch_bounds__(256) k_bwd_meta_mark(MetaArgs ma, PatchArgs a, BwdMeta* __restrict__ meta) {
    const long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (r >= a.R) return;
    const BwdMeta m = bwd_meta_of(ma, r);
    if (lane == 0) meta[r] = m;
    if (patch_area(m) == 0) return;
    const int H = a.cfg.H[m.lvl], W = a.cfg.W[m.lvl];
    unsigned* ab = a.anyb + a.word0[m.lvl];
    unsigned* mb = a.multi + a.word0[m.lvl];
    for (int y = m.y0 + lane; y <= m.y1; y += 32) {
        const long long c0 = ((long long)m.img * H + y) * W + m.x0, c1 = c0 + (m.x1 - m.x0);
        for (long long wd = c0 >> 5; wd <= (c1 >> 5); ++wd) {
            const int b0 = wd == (c0 >> 5) ? (int)(c0 & 31) : 0, b1 = wd == (c1 >> 5) ? (int)(c1 & 31) : 31;
            const unsigned bits = (b1 == 31 ? 0xffffffffu : ((1u << (b1 + 1)) - 1u)) & ~((1u << b0) - 1u);
            const unsigned old = atomicOr(ab + wd, bits);
            if (old & bits) atomicOr(mb + wd, old & bits);
        }
    }
}

__device__ __forceinline__ float4 lds128(unsigned addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}

// one row of a patch block: NR row terms in registers (no predicated slots), cells left to right; `rowmask` bit kx = the
// cell is shared with another patch (-> scratch slot), else it is written straight into the gradient map
template <int NR>
__device__ __forceinline__ void patch_row(const Term* __restrict__ rt, const Term* __restrict__ colt, const int* __restrict__ coln,
                                          unsigned sg_lane, int bw, unsigned long long rowmask, float* gcell, float* scell, int C) {
    float wy[NR > 0 ? NR : 1];
    unsigned rb[NR > 0 ? NR : 1];
#pragma unroll
    for (int i = 0; i < NR; ++i) { wy[i] = rt[i].w; rb[i] = sg_lane + (unsigned)rt[i].off; }
    for (int kx = 0; kx < bw; ++kx, gcell += C, scell += C) {
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        if (NR > 0) {
            const int nc = coln[kx];
            const Term* ct = colt + kx * kMaxTerms;
            for (int j = 0; j < nc; ++j) {
                const Term t = ct[j];
#pragma unroll
                for (int i = 0; i < NR; ++i) {
                    const float w = wy[i] * t.w;
                    const float4 g = lds128(rb[i] + (unsigned)t.off);
                    acc.x = fmaf(w, g.x, acc.x); acc.y = fmaf(w, g.y, acc.y);
                    acc.z = fmaf(w, g.z, acc.z); acc.w = fmaf(w, g.w, acc.w);
                }
            }
        }
        __stcs(reinterpret_cast<float4*>(((rowmask >> kx) & 1ull) ? scell : gcell), acc);
    }
}

__global__ void __launch_bounds__(kPT, 7) k_bwd_patch(PatchArgs a) {
    extern __shared__ __align__(16) float s_dyn[];
    if (a.flags[0]) return;
    const b2d_roi_cfg& c = a.cfg;
    const int bins = c.PH * c.PW, C = c.C;
    float* sg = s_dyn;                                               // [bins][kPPitch]
    Term* rowt = reinterpret_cast<Term*>(sg + bins * kPPitch);       // [kMaxDim][kMaxTerms]; Term.off in BYTES
    Term* colt = rowt + kMaxDim * kMaxTerms;
    int* rown = reinterpret_cast<int*>(colt + kMaxDim * kMaxTerms);
    int* coln = rown + kMaxDim;
    const long long r = blockIdx.x;
    const int cg = blockIdx.y, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const BwdMeta m = a.meta[r];
    if (patch_area(m) == 0) return;
    const int H = c.H[m.lvl], W = c.W[m.lvl];
    const int nrows = m.y1 - m.y0 + 1, ncols = m.x1 - m.x0 + 1;
    // ---- grad_out[r][cg * 128 + tid][bins] / 4 -> [bin][channel]
    {
        // the [128 channels][bins] block of this CTA is contiguous: element e = 128 i + tid, i < bins, read coalesced (a warp
        // load = 4 sectors; one thread per channel would touch 32 sectors per load and bound the kernel by L1 sector
        // requests), 16 loads in flight; the shared-memory address of e advances incrementally (e += 128: channel += 128 /
        // bins, bin += 128 % bins with one wrap)
        const float* go = gout_row(a.q, r, (long long)C * bins) + (long long)cg * kPCg * bins + tid;
        const int dch = kPT / bins, db = kPT % bins;
        const int step = db * kPPitch + dch, wrap = 1 - bins * kPPitch;
        int b = tid % bins, addr = b * kPPitch + tid / bins;
        int i = 0;
        for (; i + 16 <= bins; i += 16) {
            float v[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) v[k] = __ldg(go + (i + k) * kPT);
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                sg[addr] = v[k] * 0.25f;
                addr += step; b += db;
                if (b >= bins) { b -= bins; addr += wrap; }
            }
        }
        for (; i < bins; ++i) {
            sg[addr] = __ldg(go + i * kPT) * 0.25f;
            addr += step; b += db;
            if (b >= bins) { b -= bins; addr += wrap; }
        }
    }
    const unsigned sg_lane = (unsigned)__cvta_generic_to_shared(sg + lane * 4);
    const unsigned* mb = a.multi + a.word0[m.lvl];
    float* gl = a.grad[m.lvl] + (long long)cg * kPCg + lane * 4;
    float* sl = a.scratch + (long long)cg * kPCg + lane * 4;
    const long long p0 = a.poff[r];
    // the patch in blocks of 32 x 32 cells (one block for almost every RoI the level map places; thin RoIs clamped at the
    // image border can be a few hundred cells long)
    for (int yb = 0; yb < nrows; yb += kMaxDim) {
        for (int xb = 0; xb < ncols; xb += kMaxDim) {
            const int bh = min(kMaxDim, nrows - yb), bw = min(kMaxDim, ncols - xb);
            __syncthreads();                                         // staged gradients visible / previous block done
            // ---- weight lists: thread k < kMaxDim does block row k, thread kMaxDim + k block column k
            {
                const int ax = tid / kMaxDim, k = tid % kMaxDim;
                const int n = ax ? bw : bh;
                if (ax < 2 && k < n) {
                    const int coord = (ax ? m.x0 + xb : m.y0 + yb) + k, P = ax ? c.PW : c.PH, size = ax ? W : H;
                    const float start = ax ? m.sx : m.sy, bin = ax ? m.bw : m.bh;
                    const int step = (ax ? kPPitch : c.PW * kPPitch) * 4;
                    Term* tt = (ax ? colt : rowt) + k * kMaxTerms;
                    int cnt = 0;
                    for (int p = 0; p < P; ++p) {
                        float w = 0.0f;
                        for (int i = 0; i < 2; ++i) {
                            const AxisTap t = axis_tap(start, bin, p, i, 2, size);
                            if (t.valid) {
                                if (t.lo == coord) w += t.h;
                                if (t.hi == coord) w += t.l;
                            }
                        }
                        if (w != 0.0f) { tt[cnt].w = w; tt[cnt].off = p * step; ++cnt; }
                    }
                    (ax ? coln : rown)[k] = cnt;
                }
            }
            __syncthreads();
            for (int ky = warp; ky < bh; ky += kPT / 32) {
                const int nr = rown[ky];
                const Term* rt = rowt + ky * kMaxTerms;
                const long long cell0 = ((long long)m.img * H + (m.y0 + yb + ky)) * W + m.x0 + xb;
                // multi bits of the row's <= 64 cells
                unsigned long long rowmask;
                {
                    const long long w0 = cell0 >> 5;
                    const int sh = (int)(cell0 & 31);
                    const unsigned long long lo = (unsigned long long)__ldg(mb + w0) | ((unsigned long long)__ldg(mb + w0 + 1) << 32);
                    rowmask = lo >> sh;
                    if (sh) rowmask |= (unsigned long long)__ldg(mb + w0 + 2) << (64 - sh);
                }
                float* gcell = gl + cell0 * C;
                float* scell = sl + (p0 + (long long)(yb + ky) * ncols + xb) * C;
                switch (nr) {
                    case 0: patch_row<0>(rt, colt, coln, sg_lane, bw, rowmask, gcell, scell, C); break;
                    case 1: patch_row<1>(rt, colt, coln, sg_lane, bw, rowmask, gcell, scell, C); break;
                    case 2: patch_row<2>(rt, colt, coln, sg_lane, bw, rowmask, gcell, scell, C); break;
                    case 3: patch_row<3>(rt, colt, coln, sg_lane, bw, rowmask, gcell, scell, C); break;
                    case 4: patch_row<4>(rt, colt, coln, sg_lane, bw, rowmask, gcell, scell, C); break;
                    default:
                        for (int kx = 0; kx < bw; ++kx, gcell += C, scell += C) {
                            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
                            const int nc = coln[kx];
                            const Term* ct = colt + kx * kMaxTerms;
                            for (int j = 0; j < nc; ++j) {
                                const Term t = ct[j];
                                for (int i = 0; i < nr; ++i) {
                                    const float w = rt[i].w * t.w;
                                    const float4 g = lds128(sg_lane + (unsigned)rt[i].off + (unsigned)t.off);
                                    acc.x = fmaf(w, g.x, acc.x); acc.y = fmaf(w, g.y, acc.y);
                                    acc.z = fmaf(w, g.z, acc.z); acc.w = fmaf(w, g.w, acc.w);
                                }
                            }
                            __stcs(reinterpret_cast<float4*>(((rowmask >> kx) & 1ull) ? scell : gcell), acc);
                        }
                }
            }
        }
    }
}

__global__ void __launch_bounds__(kMThreads, 3) k_bwd_merge(PatchArgs a) {
    __shared__ int s_y0[kMCap], s_y1[kMCap], s_x0[kMCap], s_x1[kMCap];
    __shared__ long long s_po[kMCap];
    __shared__ unsigned char s_multi[kMT * kMT], s_zero[kMT * kMT];      // cells of the tile to merge / to clear
    __shared__ int s_n, s_nm, s_nz, s_warp[kMThreads / 32], s_wm[8], s_wz[8];
    if (a.flags[0]) return;
    const b2d_roi_cfg& c = a.cfg;
    const int tiles_per_img = a.tile_off[c.num_levels];
    const int img = blockIdx.x / tiles_per_img;
    int t = blockIdx.x - img * tiles_per_img, lvl = 0;
    for (int q = 1; q < c.num_levels; ++q) if (t >= a.tile_off[q]) lvl = q;
    t -= a.tile_off[lvl];
    const int H = c.H[lvl], W = c.W[lvl], C = c.C, ngroups = C / kPCg;
    const int ty0 = (t / a.tiles_x[lvl]) * kMT, tx0 = (t % a.tiles_x[lvl]) * kMT;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int* bl = a.bucket + (long long)(img * c.num_levels + lvl) * a.R;
    const int nb = a.bcount[img * c.num_levels + lvl];
    float* g = a.grad[lvl] + lane * 4;
    const float* sc = a.scratch + lane * 4;
    // ---- the tile's cells by state: thread t < 256 looks at cell (t / 16, t % 16); ordered ballot compaction, so that the
    // warps below share the cells evenly whatever their rows hold
    {
        bool isz = false, ism = false;
        if (tid < kMT * kMT) {
            const int y = ty0 + (tid >> 4), x = tx0 + (tid & 15);
            if (y < H && x < W) {
                const long long cell = ((long long)img * H + y) * W + x;
                const bool any = (__ldg(a.anyb + a.word0[lvl] + (cell >> 5)) >> (cell & 31)) & 1u;
                ism = (__ldg(a.multi + a.word0[lvl] + (cell >> 5)) >> (cell & 31)) & 1u;
                isz = !any;
            }
        }
        const unsigned bz = __ballot_sync(0xffffffffu, isz), bm = __ballot_sync(0xffffffffu, ism);
        if (lane == 0 && warp < 8) { s_wz[warp] = __popc(bz); s_wm[warp] = __popc(bm); }
        __syncthreads();
        if (warp < 8) {
            int oz = 0, om = 0;
            for (int w = 0; w < warp; ++w) { oz += s_wz[w]; om += s_wm[w]; }
            if (isz) s_zero[oz + __popc(bz & ((1u << lane) - 1u))] = (unsigned char)tid;
            if (ism) s_multi[om + __popc(bm & ((1u << lane) - 1u))] = (unsigned char)tid;
        }
        if (tid == 0) {
            int z = 0, mm = 0;
            for (int w = 0; w < 8; ++w) { z += s_wz[w]; mm += s_wm[w]; }
            s_nz = z; s_nm = mm;
        }
        __syncthreads();
    }
    const int nz = s_nz, nm = s_nm;
    for (int i = warp; i < nz; i += kMThreads / 32) {
        const int cid = s_zero[i];
        float* dst = g + (((long long)img * H + ty0 + (cid >> 4)) * W + tx0 + (cid & 15)) * C;
        for (int q = 0; q < ngroups; ++q) __stcs(reinterpret_cast<float4*>(dst + q * kPCg), make_float4(0.f, 0.f, 0.f, 0.f));
    }
    if (nm == 0) return;                                             // (uniform over the CTA)
    for (int base = 0; base == 0 || base < nb; base += kMCap) {
        // ---- RoIs of this chunk whose patch touches the tile, ascending
        {
            const int k = base + tid;
            bool hit = false;
            BwdMeta m;
            int r = 0;
            if (k < nb) {
                r = bl[k];
                m = a.meta[r];
                hit = !(m.y1 < ty0 || m.y0 > ty0 + kMT - 1 || m.x1 < tx0 || m.x0 > tx0 + kMT - 1);
            }
            const unsigned bm = __ballot_sync(0xffffffffu, hit);
            if (lane == 0) s_warp[warp] = __popc(bm);
            __syncthreads();
            int before = 0;
            for (int w = 0; w < warp; ++w) before += s_warp[w];
            if (hit) {
                const int e = before + __popc(bm & ((1u << lane) - 1u));
                s_y0[e] = m.y0; s_y1[e] = m.y1; s_x0[e] = m.x0; s_x1[e] = m.x1; s_po[e] = a.poff[r];
            }
            if (tid == 0) { int tot = 0; for (int w = 0; w < kMThreads / 32; ++w) tot += s_warp[w]; s_n = tot; }
            __syncthreads();
        }
        const int n = s_n;
        for (int i = warp; i < nm; i += kMThreads / 32) {
            const int cid = s_multi[i];
            const int y = ty0 + (cid >> 4), xx = tx0 + (cid & 15);
            float* dst = g + (((long long)img * H + y) * W + xx) * C;
            for (int e0 = 0; e0 == 0 || e0 < n; e0 += 32) {
                // lane e tests hit e0 + e and holds its scratch slot; the covering ones are visited in ascending order
                const int e = e0 + lane;
                long long slot = 0;
                bool cov = false;
                if (e < n) {
                    const int y0 = s_y0[e], x0 = s_x0[e], x1 = s_x1[e];
                    cov = y >= y0 && y <= s_y1[e] && xx >= x0 && xx <= x1;
                    slot = (s_po[e] + (long long)(y - y0) * (x1 - x0 + 1) + (xx - x0)) * C;
                }
                const unsigned mask = __ballot_sync(0xffffffffu, cov);
                const bool first = base == 0 && e0 == 0;
                for (int q = 0; q < ngroups; ++q) {
                    float4 acc = first ? make_float4(0.f, 0.f, 0.f, 0.f) : *reinterpret_cast<const float4*>(dst + q * kPCg);
                    unsigned mq = mask;
                    while (mq) {                                     // up to four slots in flight, added in order
                        float4 v[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (mq) {
                                const int src = __ffs(mq) - 1;
                                mq &= mq - 1;
                                const long long sl = __shfl_sync(0xffffffffu, slot, src);
                                v[u] = __ldcs(reinterpret_cast<const float4*>(sc + sl + q * kPCg));
                            }
                        }
#pragma unroll
                        for (int u = 0; u < 4; ++u) { acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w; }
                    }
                    *reinterpret_cast<float4*>(dst + q * kPCg) = acc;
                }
            }
        }
        __syncthreads();                                             // the hit list is rebuilt for the next chunk
    }
}

size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

long long bitmap_words(const b2d_roi_cfg& c, int B, long long* word0) {
    long long w = 0;
    for (int l = 0; l < c.num_levels; ++l) {
        if (word0) word0[l] = w;
        w += ((long long)B * c.H[l] * c.W[l] + 31) / 32;
    }
    if (word0) word0[c.num_levels] = w;
    return w;
}

}  // namespace

size_t roi_align_bwd_patch_workspace(long long R, int B, const b2d_roi_cfg& c) {
    const size_t r = (size_t)(R > 0 ? R : 1);
    const size_t words = (size_t)bitmap_words(c, B, nullptr);
    return align256(r * sizeof(BwdMeta)) + align256((size_t)B * c.num_levels * r * 4) + align256((size_t)B * c.num_levels * 4) +
           align256((r + 1) * 8) + 256 + 2 * align256(words * 4 + 16) + (size_t)patch_budget_cells(R) * c.C * 4 + 256;
}

// returns 1 if the configuration is not eligible (the caller then uses the tile / generic kernels)
int roi_align_bwd_patch_try(void* const* grad_feat_ptrs_host, const RoiSets& q, const int* levels, long long R, int B,
                            const b2d_roi_cfg& c, void* workspace, cudaStream_t st) {
    if (c.layout != 1 || c.sampling_ratio != 2 || c.PH > kMaxTerms || c.PW > kMaxTerms || c.PH * c.PW > kMaxBinsT) return 1;
    if (c.C % kPCg != 0 || R < 1) return 1;
    for (int l = 0; l < c.num_levels; ++l)
        if (reinterpret_cast<uintptr_t>(grad_feat_ptrs_host[l]) & 15) return 1;
    PatchArgs a;
    memset(&a, 0, sizeof(a));
    a.cfg = c;
    const long long words = bitmap_words(c, B, a.word0);
    char* w = (char*)workspace;
    BwdMeta* meta = (BwdMeta*)w; w += align256((size_t)R * sizeof(BwdMeta));
    int* bucket = (int*)w; w += align256((size_t)B * c.num_levels * R * 4);
    int* bcount = (int*)w; w += align256((size_t)B * c.num_levels * 4);
    long long* poff = (long long*)w; w += align256((size_t)(R + 1) * 8);
    int* flags = (int*)w; w += 256;
    unsigned* anyb = (unsigned*)w; w += align256((size_t)words * 4 + 16);
    unsigned* multi = (unsigned*)w; w += align256((size_t)words * 4 + 16);      // (+ 16: the row mask reads up to two words ahead)
    float* scratch = (float*)w;
    MetaArgs ma;
    memset(&ma, 0, sizeof(ma));
    ma.cfg = c; ma.q = q; ma.levels = levels; ma.R = R;
    a.cap_cells = patch_budget_cells(R);
    if (cudaMemsetAsync(anyb, 0, 2 * align256((size_t)words * 4 + 16), st) != cudaSuccess) return check_launch("roi_align_bwd(patch memset)");
    int run = 0;
    for (int l = 0; l < c.num_levels; ++l) {
        a.grad[l] = (float*)grad_feat_ptrs_host[l];
        a.tile_off[l] = run;
        a.tiles_x[l] = cdiv(c.W[l], kMT);
        run += a.tiles_x[l] * cdiv(c.H[l], kMT);
    }
    a.tile_off[c.num_levels] = run;
    a.q = q; a.meta = meta; a.poff = poff; a.anyb = anyb; a.multi = multi; a.scratch = scratch; a.flags = flags;
    a.bucket = bucket; a.bcount = bcount; a.R = R;
    k_bwd_meta_mark<<<cdiv(R * 32, 256), 256, 0, st>>>(ma, a, meta);
    k_bwd_bucket_scan<<<B * c.num_levels + 1, 1024, 0, st>>>(meta, R, c.num_levels, B * c.num_levels, bucket, bcount, a.cap_cells,
                                                            poff, flags);
    const size_t smem = (size_t)c.PH * c.PW * kPPitch * 4 + 2 * kMaxDim * kMaxTerms * sizeof(Term) + 2 * kMaxDim * 4;
    B2D_SMEM(k_bwd_patch, smem, "k_bwd_patch");
    k_bwd_patch<<<dim3((unsigned)R, (unsigned)(c.C / kPCg)), kPT, smem, st>>>(a);
    k_bwd_merge<<<(unsigned)(run * B), kMThreads, 0, st>>>(a);
    int rc = check_launch("roi_align_bwd(patch)");
    if (rc != B2D_OK) return rc;
    // fallback for patches that do not fit (flag raised by k_bwd_scan): the tile kernel on the same tables
    return roi_align_bwd_tile_launch(grad_feat_ptrs_host, q, R, B, c, meta, bucket, bcount, flags, st);
}

}  // namespace b2d
